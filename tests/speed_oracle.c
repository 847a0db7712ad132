/* CPU restatement of the catch-up speed control of live mode (SPEC §7.2) — TEST INFRASTRUCTURE.
 *
 * The environment oracle (oracle/abr_oracle.c) is included as it is, so the download, the pause gate, the playback
 * pieces and the reward are its own.  What §7.2 changes is where a speed comes from: the controller decides the speed
 * of a content chunk at the top of the playback loop in which the chunk starts to play.  That loop sits inside the
 * oracle's play_wall / play_content, so those two, the step that calls them and the two batch entry points are
 * restated below with the decision at that point; with the controller off (c->on = 0) they are the oracle's own
 * (tests/test_speed_oracle.py checks that bit for bit).  Built by tests/speed_oracle.py with gcc -O2
 * -ffp-contract=off -fno-fast-math (no FMA contraction), like the environment oracle.
 */
#include "../oracle/abr_oracle.c"

/* The controller of one environment: parameters {target_latency, max_drift, gain, dead_band, min_buffer}, whether it
 * is installed, the per-session decision play_speed[N] (zero at creation, untouched by resets), an optional log
 * [V][N] that receives every decision at [min(play_id, V - 1)][s], and the counts of decisions above 1, below 1 and
 * held at 1 by the buffer guard (so that a test can see its data exercise all three). */
typedef struct SpdCtl {
    double prm[5];
    int on;
    double* play_speed;
    double* log;
    int64_t count[3];
} SpdCtl;

SpdCtl* spd_create(int N) {
    SpdCtl* c = (SpdCtl*)calloc(1, sizeof(SpdCtl));
    c->play_speed = (double*)calloc((size_t)(N > 0 ? N : 1), 8);
    return c;
}

void spd_destroy(SpdCtl* c) {
    if (!c) return;
    free(c->play_speed);
    free(c);
}

/* 0 when the parameters are what abr_env_set_speed_control accepts, 1 otherwise */
int spd_params_invalid(const double* p) {
    for (int k = 0; k < 5; ++k)
        if (!isfinite(p[k])) return 1;
    if (!(p[0] >= 0.0) || !(p[1] > 0.0) || !(p[1] < 1.0) || !(p[2] > 0.0) || !(p[3] >= 0.0) || !(p[4] >= 0.0)) return 1;
    return 0;
}

/* NULL = off */
void spd_set(SpdCtl* c, const double* p) {
    c->on = p != 0;
    if (p) memcpy(c->prm, p, sizeof(c->prm));
}

void spd_set_log(SpdCtl* c, double* log) { c->log = log; }

const int64_t* spd_counts(SpdCtl* c) { return c->count; }

double* spd_play_speed(SpdCtl* c) { return c->play_speed; }

/* SPEC §7.2: the speed of a chunk that starts to play at wall clock tc with content play_time played and buffer b */
double spd_rule(const double* p, double tc, double play_time, double b) {
    double e = (tc - play_time) - p[0];
    double v;
    if (fabs(e) <= p[3]) {
        v = 1.0;
    } else {
        double y = p[2] * e;
        v = 1.0 + p[1] * (y / (1.0 + fabs(y)));
    }
    if (v > 1.0 && b < p[4]) v = 1.0;   /* never speed up into a stall */
    return v;
}

/* where §7 reads speed[min(play_id, V-1)]: the stored decision, or a new one when chunk play_id has not played yet */
static double spd_speed(OrcEnv* e, SpdCtl* c, int s, const double* speed, double tc, double b) {
    if (!c->on) return live_speed(e, s, speed);
    if (e->play_len[s] == 0.0 || !(c->play_speed[s] > 0.0)) {
        c->play_speed[s] = spd_rule(c->prm, tc, e->play_time[s], b);
        double unguarded = spd_rule(c->prm, tc, e->play_time[s], INFINITY);
        c->count[0] += c->play_speed[s] > 1.0;
        c->count[1] += c->play_speed[s] < 1.0;
        c->count[2] += unguarded > 1.0 && c->play_speed[s] == 1.0;
        if (c->log) {
            int k = e->play_id[s] < e->V ? e->play_id[s] : e->V - 1;
            c->log[(size_t)k * e->N + s] = c->play_speed[s];
        }
    }
    return c->play_speed[s];
}

/* ---- oracle/abr_oracle.c's play_wall, play_content, step_one, orc_env_step_live and orc_env_rollout_live, with the
 * speed read through spd_speed ---- */
static double spd_play_wall(OrcEnv* e, SpdCtl* c, int s, const double* speed, double* buffer, LiveAcc* a, double dt) {
    const double L = e->p.chunk_length;
    if (!e->started[s]) { a->startup = a->startup + dt; a->tc = a->tc + dt; return 0.0; }
    double rem = dt;
    while (rem > 0.0 && *buffer > 0.0) {
        double v = spd_speed(e, c, s, speed, a->tc, *buffer);
        double room = L - e->play_len[s];
        double can = room < *buffer ? room : *buffer;
        double need = v * rem;
        if (need < can) {
            live_piece(e, s, buffer, a, need, rem, v);
            e->play_len[s] = e->play_len[s] + need;
            rem = 0.0;
        } else {
            double dw = can / v;
            int finished = room <= *buffer;
            live_piece(e, s, buffer, a, can, dw, v);
            rem = rem - dw;
            if (finished) { e->play_id[s] += 1; e->play_len[s] = 0.0; }
            else e->play_len[s] = e->play_len[s] + can;
        }
    }
    if (rem < 0.0) rem = 0.0;
    a->tc = a->tc + rem;
    return rem;
}

static double spd_play_content(OrcEnv* e, SpdCtl* c, int s, const double* speed, double* buffer, LiveAcc* a, double x) {
    const double L = e->p.chunk_length;
    double w = 0.0;
    while (x > 0.0) {
        double v = spd_speed(e, c, s, speed, a->tc, *buffer);
        double room = L - e->play_len[s];
        int finished = room <= x;
        double d = finished ? room : x;
        double dw = d / v;
        live_piece(e, s, buffer, a, d, dw, v);
        w = w + dw;
        if (finished) { e->play_id[s] += 1; e->play_len[s] = 0.0; x = x - d; }
        else { e->play_len[s] = e->play_len[s] + d; x = 0.0; }
    }
    return w;
}

static void spd_step_one(OrcEnv* e, SpdCtl* c, int s, int q, const double* speed, StepOut* o) {
    const OrcParams* p = &e->p;
    memset(o, 0, sizeof(*o));
    if (e->done[s]) { o->eov = 1; o->buffer = e->buffer[s]; o->inert = 1; return; }
    const int tr = e->trace_id[s];
    const int T = e->trace_len[tr];
    const double I = e->trace_interval[tr];
    int chunk = e->chunk[s], seg = e->seg[s];
    double phi = e->phi[s], pos = e->pos[s], buffer = e->buffer[s];
    const double size = e->sizes[chunk * e->A + q];
    const double* C = e->cum + (size_t)tr * (e->T_max + 1);
    const int live = p->live != 0;
    double idle = 0.0, rebuf = 0.0, latency = 0.0;
    LiveAcc a = {0.0, 0.0, 0.0, e->t_now[s]};
    e->bad_speed = 0;
    if (live) {
        double w1 = (double)(chunk + 1) * p->chunk_length - e->t_now[s];
        w1 = max0(w1);
        rebuf = spd_play_wall(e, c, s, speed, &buffer, &a, w1);
        double w2 = (e->started[s] && buffer > p->max_buffer) ? spd_play_content(e, c, s, speed, &buffer, &a, buffer - p->max_buffer) : 0.0;
        idle = w1 + w2;
        if (idle > 0.0) { advance_trace(&seg, &phi, idle, I, T); pos = C[seg] + (C[seg + 1] - C[seg]) * phi; }
    }
    const double P = C[T];
    double delay;
    {
        double target = pos + size;
        long long n = 0;
        while (target >= P) {
            target = target - P;
            n += 1;
            if (n >= (1 << 20)) { e->errors++; target = 0.0; break; }
        }
        int j = (n == 0) ? seg : 0;
        while (j + 1 < T && C[j + 1] <= target) ++j;
        double phi_new = (target - C[j]) / (C[j + 1] - C[j]);
        long long k = (long long)(j - seg) + n * (long long)T;
        delay = max0(((double)k + (phi_new - phi)) * I) + p->rtt;
        seg = j;
        phi = phi_new;
        pos = target;
    }
    double thr = size / delay;
    double sleep = 0.0;
    if (live) {
        rebuf = rebuf + spd_play_wall(e, c, s, speed, &buffer, &a, delay);
        buffer = buffer + p->chunk_length;
        e->t_now[s] = (e->t_now[s] + idle) + delay;
        if (!e->started[s] && buffer >= p->start_up_length) e->started[s] = 1;
        latency = e->t_now[s] - e->play_time[s];
        sleep = idle;
    } else {
        rebuf = max0(delay - buffer);
        buffer = max0(buffer - delay) + p->chunk_length;
        if (buffer > p->max_buffer) {
            sleep = ceil((buffer - p->max_buffer) / p->sleep_quantum) * p->sleep_quantum;
            buffer = buffer - sleep;
            advance_trace(&seg, &phi, sleep, I, T);
            pos = C[seg] + (C[seg + 1] - C[seg]) * phi;
        }
    }
    const double u = e->util[chunk * e->A + q];
    const int lq = e->last_q[s];
    const int prow = (p->smooth_prev_ladder && chunk > 0) ? chunk - 1 : chunk;
    double smooth = (lq >= 0) ? fabs(u - e->util[prow * e->A + lq]) : 0.0;
    double reward = (u - p->rebuf_penalty * rebuf) - p->smooth_penalty * smooth;
    if (live) reward = reward - p->latency_penalty * latency;
    if (p->track_history) {
        e->bw_hist[(size_t)s * e->K + (e->hist_len[s] % e->K)] = thr;
        e->hist_len[s] += 1;
    }
    chunk += 1;
    o->delay = delay; o->sleep = sleep; o->buffer = buffer; o->rebuf = rebuf; o->reward = reward;
    o->thr = thr; o->u = u; o->smooth = smooth; o->latency = latency; o->startup = a.startup; o->area = a.area; o->played = a.played;
    if (live && e->bad_speed) e->errors++;
    o->eov = (chunk >= e->V);
    e->last_q[s] = q;
    if (o->eov && p->auto_reset) {
        chunk = 0; buffer = 0.0; e->last_q[s] = p->default_quality;
        e->hist_len[s] = 0; e->last_pred[s] = 0.0; e->err_len[s] = 0;
        e->t_now[s] = 0.0; e->play_time[s] = 0.0; e->started[s] = p->start_up_length <= 0.0;
        e->play_id[s] = 0; e->play_len[s] = 0.0;
    } else if (o->eov) {
        e->done[s] = 1;
    }
    e->chunk[s] = chunk; e->seg[s] = seg; e->phi[s] = phi; e->pos[s] = pos; e->buffer[s] = buffer;
}

void spd_env_step_live(OrcEnv* e, SpdCtl* c, const int32_t* action, const double* speed, double* delay, double* sleep,
                       double* buffer, double* rebuf, double* reward, double* latency, double* next_sizes,
                       uint8_t* eov, double* throughput, double* acc) {
    const size_t N = (size_t)e->N;
    for (int s = 0; s < e->N; ++s) {
        StepOut o;
        spd_step_one(e, c, s, action[s], speed, &o);
        if (delay) delay[s] = o.delay;
        if (sleep) sleep[s] = o.sleep;
        if (buffer) buffer[s] = o.buffer;
        if (rebuf) rebuf[s] = o.rebuf;
        if (reward) reward[s] = o.reward;
        if (latency) latency[s] = o.latency;
        if (eov) eov[s] = o.eov;
        if (throughput) throughput[s] = o.thr;
        if (next_sizes)
            for (int a = 0; a < e->A; ++a)
                next_sizes[(size_t)s * e->A + a] = e->done[s] ? 0.0 : e->sizes[e->chunk[s] * e->A + a];
        if (acc && !o.inert) {
            acc[0 * N + s] += o.reward; acc[1 * N + s] += o.rebuf; acc[2 * N + s] += o.u; acc[3 * N + s] += o.smooth;
            acc[4 * N + s] += o.sleep; acc[5 * N + s] += o.delay; acc[6 * N + s] += 1.0;
            if (o.eov) acc[7 * N + s] += 1.0;
            acc[8 * N + s] += o.startup; acc[9 * N + s] += o.area; acc[10 * N + s] += o.played;
        }
    }
}

void spd_env_rollout_live(OrcEnv* e, SpdCtl* c, int policy, uint64_t seed, int64_t session_base, int steps,
                          const int32_t* actions_in, const double* speed, double* delay, double* sleep, double* buffer,
                          double* rebuf, double* reward, double* latency, uint8_t* eov, int32_t* actions_out,
                          double* acc) {
    const int N = e->N;
    for (int s = 0; s < N; ++s) {
        double a_rew = 0, a_reb = 0, a_u = 0, a_sm = 0, a_sl = 0, a_dl = 0, a_steps = 0, a_eps = 0, a_su = 0, a_lat = 0, a_pl = 0;
        for (int t = 0; t < steps; ++t) {
            int q = policy_action(e, s, policy, seed, session_base, t, actions_in);
            StepOut o;
            size_t ix = (size_t)t * N + s;
            spd_step_one(e, c, s, q, speed, &o);
            if (delay) delay[ix] = o.delay;
            if (sleep) sleep[ix] = o.sleep;
            if (buffer) buffer[ix] = o.buffer;
            if (rebuf) rebuf[ix] = o.rebuf;
            if (reward) reward[ix] = o.reward;
            if (latency) latency[ix] = o.latency;
            if (eov) eov[ix] = o.eov;
            if (actions_out) actions_out[ix] = q;
            if (!o.inert) {
                a_rew = a_rew + o.reward; a_reb = a_reb + o.rebuf; a_u = a_u + o.u;
                a_sm = a_sm + o.smooth; a_sl = a_sl + o.sleep; a_dl = a_dl + o.delay;
                a_su = a_su + o.startup; a_lat = a_lat + o.area; a_pl = a_pl + o.played;
                a_steps += 1.0; if (o.eov) a_eps += 1.0;
            }
        }
        if (acc) {
            acc[0 * (size_t)N + s] = a_rew; acc[1 * (size_t)N + s] = a_reb; acc[2 * (size_t)N + s] = a_u;
            acc[3 * (size_t)N + s] = a_sm; acc[4 * (size_t)N + s] = a_sl; acc[5 * (size_t)N + s] = a_dl;
            acc[6 * (size_t)N + s] = a_steps; acc[7 * (size_t)N + s] = a_eps;
            acc[8 * (size_t)N + s] = a_su; acc[9 * (size_t)N + s] = a_lat; acc[10 * (size_t)N + s] = a_pl;
        }
    }
    e->step_base += (uint32_t)(steps > 0 ? steps : 0);
}
