// Chunk-step kernels (SPEC.md §2-§4, §6, §7): one thread per session.
//
// Replaces the per-session fixed-dt Python loop of the reference (Simulator.py:135-208: download block
// :152-170, playback/buffer block :137-140,174-202, pause gate :143-145) with a closed form over the
// square-wave trace (NetworkInfo, Simulator.py:37-42).
//
//  * abr_step_kernel     one chunk step per launch, SoA state in HBM (RL harness form).  HBM-bound:
//                        44 B read + 36 B state write + 41 B outputs per session-step (DESIGN.md §4).
//  * abr_rollout_kernel  `steps` chunk steps per launch with the state in registers and the trajectory
//                        streamed out with st.global.cs (41 B/step) — the fused-episode form.
//  * abr_trace_table_kernel, abr_reset_kernel, abr_stats_* helpers.
//
// SPEC §3.1 integrates the download against the trace's cumulative capacity C[j] (data deliverable from the
// start of the trace period up to the start of segment j, accumulated left to right once per environment).  A
// session carries its position in those data coordinates (`pos`), so a download is `target = pos + size`
// followed by "which segment holds `target`" — and, as long as the session does not sleep, the next download's
// target does not depend on anything this step computes after that one addition.  The step is therefore split in
// two halves:
//   head  target -> segment j with C[j] <= target < C[j+1], through the per-trace bucket index (abr_common.cuh:
//         one 16-bit pair lookup bounds j to a handful of candidates — none or one on typical traces — that are
//         settled with exact compares on C); a fixed, branch-free sequence in the common case.
//   tail  the division that turns the position inside segment j into time, delay, buffer drain / rebuffer,
//         sleep cap, reward, stores.
// The fused episode issues the head of step t+1 *before* the tail of step t (software pipelining: two independent
// instruction streams per thread instead of one serial chain) and redoes it in the rare case that step t slept.
// Two access paths for C and the index:
//   * shared-memory path (both kernels): when all sessions of a thread block (a 128-session tile in the per-step
//     kernel) follow the same trace and its rows fit, the block stages them in shared memory with TMA bulk
//     copies and every probe is an LDS — the "traces staged in shared memory" design of the north star.
//   * global path (any session order): read-only loads (ld.global.nc): one 32-byte record, one index pair and
//     one or two sectors of C per step; the tables (25 MB at the benchmark shape) are L2-resident.
#include <type_traits>

#include "abr_common.cuh"
#include "../../include/abr_b200_dynamic.h"

namespace abr {

namespace {

constexpr int kStepBlock = 256;      // helper kernels (reset, tables, cost)
#ifndef ABR_STEP_PF_DIST
#define ABR_STEP_PF_DIST 2           // the per-step kernel asks the tile this many tiles ahead into L2 (1: off)
#endif
// The per-step kernel's L2 prefetch is for batches that stream from HBM: state + outputs (121 B per session) well
// beyond the 126 MB L2.  A batch that lives in L2 from one step to the next (back-to-back steps of 524 288 or 1 Mi
// sessions) only pays for the instructions: 18.4 -> 20.5 us and 24.7 -> 26.2 us.
constexpr long long kPrefetchMinBytes = 192ll << 20;
constexpr int kTile = 128;           // threads per block = sessions per tile of the per-step kernel
constexpr int kTileBlocksPerSM = 7;
constexpr int kStepTiles = 8;         // least number of tiles per block of the per-step kernel
constexpr int kRolloutBlock = 64;   // 65 536 sessions -> 1 024 blocks = 6.9 per SM (balanced over 148 SMs)
constexpr int kStatsBlock = 256;
constexpr int kStatsSessionsPerBlock = 1024;   // 64 blocks at 65 536 sessions: enough loads in flight to hide HBM latency
constexpr int kWrapGuard = 1 << 20;            // safety net of the whole-period loop (SPEC §3.1)
#ifndef ABR_ROLLOUT_UNROLL
#define ABR_ROLLOUT_UNROLL 1   // A/B-tested on B200: 1 and 2 are within 0.3 % of each other; 1 is half the code and spills nothing
#endif
constexpr int kRolloutUnroll = ABR_ROLLOUT_UNROLL;   // steps per trip of the fused episode's loop

struct Sess {
    const double* __restrict__ cum;    // C[0..T] of the session's trace (global row)
    const uint16_t* __restrict__ idx;  // bucket index of the session's trace (global row)
    uint32_t cum_s, idx_s, tab_s;      // shared-memory addresses of the block's copies (SMEM path)
    const double2* __restrict__ tab;   // [V][A] {chunk size, utility} (global table)
    double I, phi, buffer;             // phi = fraction of segment `seg` already consumed (SPEC §1)
    double inv_I;                      // pow2_inverse(I): 1/I when that is exact, else 0 (the sleeping step's chain starts with it)
    double pos;                        // the same position in data coordinates: C[seg] + (C[seg+1] - C[seg]) * phi
    double P, scale;                   // C[T]: capacity of one trace period; cells per unit of data
    double Td;                         // (double)T
    int T, M, seg, chunk, last_q, hist_len;
    bool done;
    // live mode (SPEC §7)
    double t_now, play_time, play_len;   // wall clock, content played, content played of the chunk being played
    const double* __restrict__ speed;    // playback speed of content chunk k at speed[k * speed_stride] (null = 1.0)
    size_t speed_stride;
    double play_speed;                   // LIVE = 2 (SPEC §7.2): the speed decided for chunk play_id
    const EnvView::SpeedControl* ctl;    // LIVE = 2: the controller's parameters
    int play_id, V;                      // content chunk being played
    bool started, bad_speed;
#ifdef ABR_CHECKED
    int chk_cum_n, chk_idx_n, chk_tab_n;  // entries the C row / index row / {size, utility} table may be read at
#endif
};

struct StepRes {
    double delay, sleep, buffer, rebuf, reward, thr, u, smooth, latency, startup, area, played;
    bool eov, inert, walk_error, reset_mpc;
};

__device__ __forceinline__ uint32_t lds_u16(uint32_t addr) {
    uint32_t x;
    asm volatile("ld.shared.u16 %0, [%1];" : "=r"(x) : "r"(addr));
    return x;
}

__device__ __forceinline__ double lds_f64(uint32_t addr) {
    double x;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(x) : "r"(addr));
    return x;
}

__device__ __forceinline__ double2 lds_f64x2(uint32_t addr) {
    double2 x;
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(x.x), "=d"(x.y) : "r"(addr));
    return x;
}

// Cell of a data position in the bucket index: x * scale rounded to the nearest integer, clamped to M - 1.  The
// rounding goes through the 2^52 trick (the low word of x*scale + 1.5*2^52 is the integer for 0 <= x*scale < 2^31):
// one FP64 add (8 cycles) instead of a conversion instruction on the slow XU pipe.  Non-decreasing in x, which is all
// the index needs (abr_common.cuh); the table is built with this same function.
__device__ __forceinline__ uint32_t cell_of(const double x, const double scale, const int M) {
    const double y = dadd(dmul(x, scale), 6755399441055744.0);
    return min((uint32_t)__double2loint(y), (uint32_t)(M - 1));
}

// (double)(a - b) for |a - b| < 2^31, exact, without the XU conversion: 2^52 + 2^31 + i has i + 2^31 in its low word;
// the bias is folded into the subtraction (one three-input integer add)
__device__ __forceinline__ double diff2double(const int a, const int b) {
    return dsub(__hiloint2double(0x43300000, (int)((uint32_t)a - (uint32_t)b + 0x80000000u)), 4503601774854144.0);
}

// max(x, 0) = (x + |x|) / 2 on the FP64 pipe: exact (x + x and the halving never round; x - x = +0), two dependent
// FP64 operations (16 cycles) where the sign-mask form of abr_common.cuh takes three on the busier integer pipe.
__device__ __forceinline__ double max0d(double x) { return dmul(dadd(x, fabs(x)), 0.5); }

// One aligned 256-bit read-only load (SASS LDG.E.256): a scattered load costs the L1 one tag cycle per distinct line
// whatever its width, so the global path fetches four doubles per instruction.
struct Quad { double a, b, c, d; };
__device__ __forceinline__ Quad ldg256(const void* p) {
    Quad q;
    asm("ld.global.nc.v4.f64 {%0, %1, %2, %3}, [%4];" : "=d"(q.a), "=d"(q.b), "=d"(q.c), "=d"(q.d) : "l"(p));
    return q;
}

// x[k] of eight doubles held in registers, k in [0, 8): a three-level select tree.
__device__ __forceinline__ double sel8(const Quad& A, const Quad& B, const int k) {
    const bool b0 = (k & 1) != 0, b1 = (k & 2) != 0, b2 = (k & 4) != 0;
    const double y0 = b0 ? A.b : A.a, y1 = b0 ? A.d : A.c, y2 = b0 ? B.b : B.a, y3 = b0 ? B.d : B.c;
    const double z0 = b1 ? y1 : y0, z1 = b1 ? y3 : y2;
    return b2 ? z1 : z0;
}

// C[j] / idx[b] of the session's trace: an LDS on the shared-memory path, else a read-only global load.
template <bool SMEM>
__device__ __forceinline__ double ld_c(const Sess& s, const int j) {
    ABR_CHECK(j >= 0 && j < s.chk_cum_n, "C row index");
    return SMEM ? lds_f64(s.cum_s + 8u * (uint32_t)j) : __ldg(s.cum + j);
}

template <bool SMEM>
__device__ __forceinline__ int ld_idx(const Sess& s, const int b) {
    ABR_CHECK(b >= 0 && b < s.chk_idx_n, "bucket index entry");
    return SMEM ? (int)lds_u16(s.idx_s + 2u * (uint32_t)b) : (int)__ldg(s.idx + b);
}

// The table reads of one step (SPEC §3.1 size, §3.4 utilities).  They depend only on (chunk, q, last_q), so the fused
// episode issues them ahead of the step.
struct Lookup { double size, u, u_prev; };

// prev_ladder (AbrParams.smooth_prev_ladder): the previous quality is looked up in the previous chunk's own ladder
// (Simulator.calculate_qoe, Simulator.py:81-82) instead of the current chunk's (mpc.py:148-149).
template <bool SMEM>
__device__ __forceinline__ Lookup lookup_tables(const Sess& s, const int A, const int V, const int chunk, const int q,
                                                const int last_q, const bool prev_ladder) {
    const int row = (chunk < V ? chunk : 0) * A;   // an inert session (chunk == V) reads row 0 and ignores it
    const int prow = (prev_ladder && last_q >= 0 && chunk > 0 && chunk < V) ? row - A : row;
    Lookup k;
    ABR_CHECK(row + q >= 0 && row + q < s.chk_tab_n && q >= 0, "{size, utility} table entry");
    ABR_CHECK(prow + (last_q >= 0 ? last_q : q) >= 0 && prow + (last_q >= 0 ? last_q : q) < s.chk_tab_n, "previous-quality table entry");
    const double2 su = SMEM ? lds_f64x2(s.tab_s + 16u * (uint32_t)(row + q)) : __ldg(s.tab + row + q);
    k.size = su.x;
    k.u = su.y;
    // no previous chunk (last_q < 0): the smoothness term |u - u_prev| is 0
    const int lq = last_q >= 0 ? last_q : q;
    k.u_prev = SMEM ? lds_f64(s.tab_s + 16u * (uint32_t)(prow + lq) + 8u) : __ldg(&s.tab[prow + lq].y);
    return k;

}

// SPEC §3.3: move the trace position forward by dt seconds without downloading.
__device__ __forceinline__ void advance_trace(int& seg, double& phi, const double dt, const double I, const double inv_i,
                                              const int T) {
    // x / d == x * (1/d) bit for bit when d is a power of two (barring over/underflow, excluded by the range check in
    // pow2_inverse), which saves the division for the usual 0.5 s / 1 s intervals; inv_i = pow2_inverse(I)
    const double x = dadd(phi, inv_i != 0.0 ? dmul(dt, inv_i) : ddiv(dt, I));
    const double n = floor(x);
    phi = dsub(x, n);          // exact, in [0, 1)
    if (n < 2147480000.0) {    // 32-bit fast path; the modulo only runs when the position wraps
        const unsigned tot = (unsigned)seg + (unsigned)(int)n;
        seg = tot >= (unsigned)T ? (int)(tot % (unsigned)T) : (int)tot;
    } else {
        seg = (int)(((long long)seg + (long long)fmod(n, (double)T)) % (long long)T);
    }
}

// SPEC §3.1 / §3.3: data-space position of (seg, phi).
template <bool SMEM>
__device__ __forceinline__ double position_of(const Sess& s, const int seg, const double phi) {
    const double c0 = ld_c<SMEM>(s, seg), c1 = ld_c<SMEM>(s, seg + 1);
    return dadd(c0, dmul(dsub(c1, c0), phi));
}

// ---- SPEC §7 playback model (live mode): the closed form of the reference's playback block, Simulator.py:174-187 ----
// The playback speed belongs to the content chunk being played (speed_controller.get_next_speed() is called when a
// chunk starts to play, Simulator.py:176-177), so playback over a wall-clock interval is piecewise: one stretch per
// content chunk.  `area` integrates the latency (wall clock - content played) over the stretches: the reference's
// average_latency is that integral per tick (Simulator.py:179-180, see SPEC §7).
struct LiveAcc { double startup, area, played, tc; };   // tc: wall clock inside the step

// LIVE: 1 = the speeds come from the caller's [V][N] table, 2 = the catch-up controller of SPEC §7.2 decides the speed
// of a chunk when it starts to play, from the latency at wall clock tc and the buffer at that instant.
template <int LIVE>
__device__ __forceinline__ double live_speed(Sess& s, const double tc, const double buffer) {
    if constexpr (LIVE == 2) {
        if (s.play_len == 0.0 || !(s.play_speed > 0.0)) {   // chunk play_id has not played yet, or no decision is stored
            const EnvView::SpeedControl& c = *s.ctl;
            const double e = dsub(dsub(tc, s.play_time), c.target_latency);
            double v = 1.0;
            if (!(fabs(e) <= c.dead_band)) {
                const double y = dmul(c.gain, e);
                v = dadd(1.0, dmul(c.max_drift, ddiv(y, dadd(1.0, fabs(y)))));
            }
            if (v > 1.0 && buffer < c.min_buffer) v = 1.0;   // never speed up into a stall
            s.play_speed = v;
        }
        return s.play_speed;
    } else {
        if (!s.speed) return 1.0;
        const int k = s.play_id < s.V ? s.play_id : s.V - 1;
        ABR_CHECK(k >= 0 && k < s.V, "playback-speed table row");
        double v = __ldg(s.speed + (size_t)k * s.speed_stride);
        if (!(v > 0.0)) { s.bad_speed = true; v = 1.0; }
        return v;
    }
}

// one stretch: d seconds of content in dw seconds of wall time at speed v
__device__ __forceinline__ void live_piece(Sess& s, double& buffer, LiveAcc& a, const double d, const double dw,
                                           const double v) {
    a.area = dadd(a.area, dadd(dmul(dsub(a.tc, s.play_time), dw), dmul(dmul(dsub(1.0, v), dw), dmul(dw, 0.5))));
    s.play_time = dadd(s.play_time, d);
    buffer = dsub(buffer, d);
    a.tc = dadd(a.tc, dw);
    a.played = dadd(a.played, d);
}

// playback during dt seconds of wall time; returns the stall time
template <int LIVE>
__device__ __forceinline__ double live_play_wall(Sess& s, double& buffer, LiveAcc& a, const double dt, const double L) {
    if (!s.started) { a.startup = dadd(a.startup, dt); a.tc = dadd(a.tc, dt); return 0.0; }
    double rem = dt;
    while (rem > 0.0 && buffer > 0.0) {
        const double v = live_speed<LIVE>(s, a.tc, buffer);
        const double room = dsub(L, s.play_len);
        const double can = room < buffer ? room : buffer;
        const double need = dmul(v, rem);
        if (need < can) {
            live_piece(s, buffer, a, need, rem, v);
            s.play_len = dadd(s.play_len, need);
            rem = 0.0;
        } else {
            const double dw = ddiv(can, v);
            const bool finished = room <= buffer;          // the chunk ends before the buffer does
            live_piece(s, buffer, a, can, dw, v);
            rem = dsub(rem, dw);
            if (finished) { s.play_id += 1; s.play_len = 0.0; }
            else s.play_len = dadd(s.play_len, can);
        }
    }
    if (rem < 0.0) rem = 0.0;
    a.tc = dadd(a.tc, rem);
    return rem;
}

// playback until x seconds of content have drained (x <= buffer); returns the wall time it takes
template <int LIVE>
__device__ __forceinline__ double live_play_content(Sess& s, double& buffer, LiveAcc& a, double x, const double L) {
    double w = 0.0;
    while (x > 0.0) {
        const double v = live_speed<LIVE>(s, a.tc, buffer);
        const double room = dsub(L, s.play_len);
        const bool finished = room <= x;
        const double d = finished ? room : x;
        const double dw = ddiv(d, v);
        live_piece(s, buffer, a, d, dw, v);
        w = dadd(w, dw);
        if (finished) { s.play_id += 1; s.play_len = 0.0; x = dsub(x, d); }
        else { s.play_len = dadd(s.play_len, d); x = 0.0; }
    }
    return w;
}

// ---- head of a step (SPEC §3.1): where does the download end? ----
// target is the wrapped data position in [0, P), kx = n*T as a double (n = whole trace periods the download went
// through), j the segment with C[j] <= target < C[j+1], c_j / c_j1 those two entries.
struct Head { double target, c_j, c_j1, kx; int j; };

// Common case as one branch-free sequence: at most one wrap, and the target's cell holds at most three segment
// boundaries.  Returns false otherwise (the caller then runs head_any); the loads are in range either way.
// Needs an index (s.M > 0).  Three dependent rounds of loads: the index pair, the candidate boundaries, C[j] / C[j+1].
template <bool SMEM>
__device__ __forceinline__ bool head_fast(const Sess& s, const double raw, Head& h) {
    const bool w = raw >= s.P;
    const double t = w ? dsub(raw, s.P) : raw;
    const uint32_t b = cell_of(t, s.scale, s.M);
    const int j0 = ld_idx<SMEM>(s, (int)b);
    int j;
    bool ok;
    if (SMEM) {
        // The index guarantees C[j0] <= t and that every boundary above idx[b + 1] lies beyond t; C is increasing, so
        // the boundaries <= t among C[j0 + 1 .. j0 + 3] are a prefix and their count places j without looking at
        // idx[b + 1] at all.  Whether three candidates were enough is checked on the result itself: t < C[j + 1]
        // (entries past C[T] are +inf, the staged row carries the slack the unconditional reads need).
        const double c1 = ld_c<SMEM>(s, j0 + 1), c2 = ld_c<SMEM>(s, j0 + 2), c3 = ld_c<SMEM>(s, j0 + 3);
        j = j0 + (c1 <= t ? 1 : 0) + (c2 <= t ? 1 : 0) + (c3 <= t ? 1 : 0);
        h.c_j = ld_c<SMEM>(s, j);                // a third round of (cheap) shared-memory loads instead of selects
        h.c_j1 = ld_c<SMEM>(s, j + 1);
        ok = t < h.c_j1;
    } else {
        // Global path: bound by the L1's tag stage (one cycle per lane and scattered load instruction), and every
        // dependent round is an L2 round trip.  So: one index entry, then the aligned eight-entry window of C that
        // holds C[j0] as two 256-bit loads.  C[q0 .. j0] <= t by the index, entries past the row's C[T] are +inf,
        // and C is increasing, so the entries <= t are a prefix of the window and their count places j — provided
        // C[j+1] is still inside the window (count <= 7).
        const int q0 = j0 & ~3;
        ABR_CHECK(q0 >= 0 && q0 + 8 <= s.chk_cum_n, "eight-entry window of C");
        const Quad A = ldg256(s.cum + q0), B = ldg256(s.cum + q0 + 4);
        const int n_le = (A.a <= t ? 1 : 0) + (A.b <= t ? 1 : 0) + (A.c <= t ? 1 : 0) + (A.d <= t ? 1 : 0) +
                         (B.a <= t ? 1 : 0) + (B.b <= t ? 1 : 0) + (B.c <= t ? 1 : 0) + (B.d <= t ? 1 : 0);
        ok = n_le >= 1 && n_le <= 7;
        const int i = ok ? n_le - 1 : 0;
        j = q0 + i;
        h.c_j = sel8(A, B, i);
        h.c_j1 = sel8(A, B, i + 1);
    }
    h.target = t;
    h.j = j;
    h.kx = w ? s.Td : 0.0;
    return ok && t < s.P;
}

// Any case: several whole-period wraps, any number of boundaries in the cell, traces without an index (bisection).
template <bool SMEM>
__device__ __forceinline__ void head_any(const Sess& s, double target, Head& h, bool& walk_error) {
    int n = 0;
    if (target >= s.P) {
        do { target = dsub(target, s.P); ++n; } while (target >= s.P && n < kWrapGuard);
        if (n >= kWrapGuard) { walk_error = true; target = 0.0; }
    }
    int j, j_hi;
    if (s.M > 0) {
        const uint32_t b = cell_of(target, s.scale, s.M);
        j = ld_idx<SMEM>(s, (int)b);
        j_hi = ld_idx<SMEM>(s, (int)b + 1);
    } else {
        j = 0;
        j_hi = s.T - 1;
    }
    if (j_hi - j > 8) {   // long run of candidates (a stretch of near-zero bandwidth, or no index): bisection
        while (j < j_hi) {
            const int mid = (j + j_hi + 1) >> 1;
            if (ld_c<SMEM>(s, mid) <= target) j = mid; else j_hi = mid - 1;
        }
    }
    double c_j = ld_c<SMEM>(s, j), c_j1 = ld_c<SMEM>(s, j + 1);
    while (j < j_hi && c_j1 <= target) { ++j; c_j = c_j1; c_j1 = ld_c<SMEM>(s, j + 1); }
    if (!(target < c_j1)) walk_error = true;       // insurance: the candidates covered the download (head_fast
                                                   // only reports success when they did)
    h.target = target; h.j = j; h.c_j = c_j; h.c_j1 = c_j1;
    h.kx = n == 0 ? 0.0 : dmul((double)n, s.Td);   // exact in fp64
}

template <bool SMEM>
__device__ __forceinline__ void head(const Sess& s, const double raw, Head& h, bool& walk_error) {
    if (s.M == 0 || !head_fast<SMEM>(s, raw, h)) head_any<SMEM>(s, raw, h, walk_error);
}

// SPEC §7.1 pause gate (Simulator.py:143-145): wait for the live edge, then for room in the buffer; moves the trace
// position by the idle time.  Runs before the head of a live step.
struct LiveGate { double buffer, rebuf, idle; LiveAcc a; };

template <bool SMEM, int LIVE>
__device__ __forceinline__ void live_gate(const EnvView& v, Sess& s, LiveGate& g) {
    const AbrParams& p = v.p;
    g.buffer = s.buffer;
    g.a.startup = g.a.area = g.a.played = 0.0;
    g.a.tc = s.t_now;
    const double w1 = max0(dsub(dmul((double)(s.chunk + 1), p.chunk_length), s.t_now));
    g.rebuf = live_play_wall<LIVE>(s, g.buffer, g.a, w1, p.chunk_length);
    const double w2 = (s.started && g.buffer > p.max_buffer)
                          ? live_play_content<LIVE>(s, g.buffer, g.a, dsub(g.buffer, p.max_buffer), p.chunk_length) : 0.0;
    g.idle = dadd(w1, w2);
    if (g.idle > 0.0) {
        advance_trace(s.seg, s.phi, g.idle, s.I, s.inv_I, s.T);
        s.pos = position_of<SMEM>(s, s.seg, s.phi);
    }
}

// ---- tail of a step (SPEC §3.1 from the division on, §3.2-§3.5) for one session held in registers ----
// `q` must already be a valid index; `lk` holds the step's table reads, `h` its head.
// FAST: auto_reset is on (a session is never inert) — drops the done/inert bookkeeping.
// LIVE: live-streaming semantics of SPEC §7 (`g` = the step's pause gate); 2 = with the speed controller of §7.2.
// Returns true when the step moved the trace position in time (sleep): s.pos was then recomputed from (seg, phi)
// and a head issued ahead for the next step is stale.
// `p` / `V`: the environment's parameters and chunk count; inv_q = pow2_inverse(p.sleep_quantum).
template <bool SMEM, bool FAST, int LIVE>
__device__ __forceinline__ bool step_tail(const AbrParams& p, const int V, Sess& s, const Head& h, const int q,
                                          const Lookup& lk, const LiveGate& g, StepRes& r, const bool want_thr,
                                          const double inv_q) {
    r.reset_mpc = false;
    if (!FAST && s.done) {  // only reachable with auto_reset == 0
        r.delay = r.sleep = r.rebuf = r.reward = r.thr = r.u = r.smooth = r.latency = r.startup = r.area = r.played = 0.0;
        r.buffer = s.buffer;
        r.eov = true;
        r.inert = true;
        return false;
    }
    r.inert = false;
    const double size = lk.size, u = lk.u, u_prev = lk.u_prev;
    const int T = s.T;
    // segment boundaries crossed: (j - seg) + n*T (both terms and the sum are exact)
    const double kd = dadd(diff2double(h.j, s.seg), h.kx);
    const double phi_new = ddiv(dsub(h.target, h.c_j), dsub(h.c_j1, h.c_j));   // fraction of segment j consumed
    const double delay = dadd(max0d(dmul(dadd(kd, dsub(phi_new, s.phi)), s.I)), p.rtt);
    int seg = h.j;
    double phi = phi_new;
    bool moved = false;
    r.thr = want_thr ? ddiv(size, delay) : 0.0;
    double rebuf, buffer, sleep = 0.0;
    r.latency = 0.0;
    r.startup = r.area = r.played = 0.0;
    s.pos = h.target;
    if (LIVE) {   // 7.2
        double live_buffer = g.buffer;
        LiveAcc a = g.a;
        rebuf = dadd(g.rebuf, live_play_wall<LIVE>(s, live_buffer, a, delay, p.chunk_length));
        buffer = dadd(live_buffer, p.chunk_length);
        s.t_now = dadd(dadd(s.t_now, g.idle), delay);
        if (!s.started && buffer >= p.start_up_length) s.started = true;
        r.latency = dsub(s.t_now, s.play_time);
        r.startup = a.startup; r.area = a.area; r.played = a.played;
        sleep = g.idle;
    } else {
        // 3.2 buffer drain / rebuffer
        // max(delay - buffer, 0) and max(buffer - delay, 0) from one subtraction: buffer - delay is exactly
        // -(delay - buffer) and at most one of the two is positive, so both are sign-masked copies of the difference
        // (five integer operations instead of five more on the FP64 pipe, whose instructions issue at half rate)
        {
            const double d = dsub(delay, s.buffer);
            const int hi = __double2hiint(d), lo = __double2loint(d);
            const int neg = hi >> 31;                      // all ones when the buffer outlasts the download
            rebuf = __hiloint2double(hi & ~neg, lo & ~neg);
            buffer = dadd(__hiloint2double((hi ^ (int)0x80000000u) & neg, lo & neg), p.chunk_length);
        }
        // 3.3 sleep cap
        if (buffer > p.max_buffer) {
            const double over = dsub(buffer, p.max_buffer);
            sleep = dmul(ceil(inv_q != 0.0 ? dmul(over, inv_q) : ddiv(over, p.sleep_quantum)), p.sleep_quantum);
            buffer = dsub(buffer, sleep);
            advance_trace(seg, phi, sleep, s.I, s.inv_I, T);
            s.pos = position_of<SMEM>(s, seg, phi);
            moved = true;
        }
    }
    // 3.4 reward
    const double smooth = fabs(dsub(u, u_prev));   // u_prev == u when there is no previous chunk (lookup_tables)
    r.reward = dsub(dsub(u, dmul(p.rebuf_penalty, rebuf)), dmul(p.smooth_penalty, smooth));
    if (LIVE) r.reward = dsub(r.reward, dmul(p.latency_penalty, r.latency));
    r.delay = delay; r.sleep = sleep; r.buffer = buffer; r.rebuf = rebuf; r.u = u; r.smooth = smooth;
    // 3.5 advance
    s.hist_len += 1;
    s.last_q = q;
    s.chunk += 1;
    s.seg = seg;
    s.phi = phi;
    s.buffer = buffer;
    r.eov = (s.chunk >= V);
    if (r.eov) {
        if (FAST || p.auto_reset) {
            s.chunk = 0; s.buffer = 0.0; s.last_q = p.default_quality; s.hist_len = 0;
            if (LIVE) { s.t_now = 0.0; s.play_time = 0.0; s.play_len = 0.0; s.play_id = 0; s.started = p.start_up_length <= 0.0; }
            r.reset_mpc = true;
        } else {
            s.done = true;
        }
    }
    return moved;
}

// One whole step (gate, head, tail) — the per-step kernel's form.
template <bool SMEM, bool FAST, int LIVE>
__device__ __forceinline__ void step_core(const EnvView& v, Sess& s, const int q, const Lookup& lk, StepRes& r,
                                          const bool want_thr) {
    r.walk_error = false;
    LiveGate g;
    g.buffer = s.buffer; g.rebuf = g.idle = 0.0;
    g.a.startup = g.a.area = g.a.played = g.a.tc = 0.0;
    Head h;
    if (!FAST && s.done) {
        h.target = h.c_j = h.kx = 0.0; h.c_j1 = 1.0; h.j = 0;
    } else {
        if (LIVE) live_gate<SMEM, LIVE>(v, s, g);
        head<SMEM>(s, dadd(s.pos, lk.size), h, r.walk_error);
    }
    step_tail<SMEM, FAST, LIVE>(v.p, v.V, s, h, q, lk, g, r, want_thr, pow2_inverse(v.p.sleep_quantum));
}

// The knobs of the policy rules below: a session's (SPEC §4.7) or the environment-wide ones.  session_knobs: session
// c's row of the per-session table, c being the caller's index of the session (the parameters are keyed like the draws
// of §8); only the fields policy P reads are loaded.
struct SessKnobs { double bba_reservoir, bba_cushion, rb_safety, bola_Vp, bola_gp, dyn_on, dyn_off; };

template <int P>
__device__ __forceinline__ SessKnobs session_knobs(const EnvView& v, const int i) {
    const int c = v.perm ? __ldg(v.perm + i) : i;
    const double* __restrict__ t = v.sp.tab + c;
    const size_t cap = (size_t)v.cap;
    SessKnobs k{};
    if (P == ABR_POLICY_BBA) { k.bba_reservoir = __ldg(t + kSpBbaReservoir * cap); k.bba_cushion = __ldg(t + kSpBbaCushion * cap); }
    if (P == ABR_POLICY_RATE || P == ABR_POLICY_DYNAMIC) k.rb_safety = __ldg(t + kSpRbSafety * cap);
    if (P == ABR_POLICY_BOLA || P == ABR_POLICY_DYNAMIC) { k.bola_Vp = __ldg(t + kSpBolaVp * cap); k.bola_gp = __ldg(t + kSpBolaGp * cap); }
    if (P == ABR_POLICY_DYNAMIC) { k.dyn_on = __ldg(t + kSpSwitchOn * cap); k.dyn_off = __ldg(t + kSpSwitchOff * cap); }
    return k;
}

// The environment-wide knobs, all seven: kernel parameters, so a field no rule of the caller reads is never loaded.
__device__ __forceinline__ SessKnobs env_knobs(const EnvView& v) {
    return SessKnobs{v.p.bba_reservoir, v.p.bba_cushion, v.pol.rb_safety, v.pol.bola_Vp, v.pol.bola_gp, v.pol.dyn_on,
                     v.pol.dyn_off};
}

// SPEC §4, buffer-based policy on the pre-step buffer level.
__device__ __forceinline__ int policy_bba(const EnvView& v, const SessKnobs& k, const double b) {
    const int A = v.A;
    if (b < k.bba_reservoir) return 0;
    if (b >= dadd(k.bba_reservoir, k.bba_cushion)) return A - 1;
    const int q = (int)floor(ddiv(dmul((double)(A - 1), dsub(b, k.bba_reservoir)), k.bba_cushion));
    return q > A - 1 ? A - 1 : q;
}

// SPEC §4.2, rate-based policy: the highest quality whose size fits rb_safety * (harmonic mean of the last
// min(hist_len, K) throughput samples) * L.  Session i's ring is column i of bw_hist[K][cap], newest sample at slot
// (hist_len - 1) mod K; it is read with plain loads (the fused episode writes it as it goes).  size_at(a): the size of
// quality a of the session's current chunk.
template <typename SizeAt>
__device__ __forceinline__ int policy_rate(const EnvView& v, const SessKnobs& k, const int i, const int hist_len,
                                           const SizeAt& size_at) {
    const int A = v.A, K = v.K;
    const int n = hist_len < K ? hist_len : K;
    if (n == 0) {
        const int d = v.p.default_quality;
        return d < 0 ? 0 : (d > A - 1 ? A - 1 : d);
    }
    double S = 0.0;
    for (int j = 0; j < n; ++j) {   // oldest first
        const int slot = (hist_len - n + j) % K;
        S = dadd(S, ddiv(1.0, v.bw_hist[(size_t)slot * v.cap + i]));
    }
    const double budget = dmul(dmul(k.rb_safety, ddiv((double)n, S)), v.p.chunk_length);
    int q = 0;
    for (int a = 0; a < A; ++a)
        if (size_at(a) <= budget) q = a;   // a NaN budget fits nothing
    return q;
}

// SPEC §4.3, BOLA: the first quality of the largest score (Vp * (v[chunk][a] + gp) - buffer) / size[chunk][a] on the
// pre-step buffer b; v is the host-built log table (bola_v, read-only path).  row: first element of the chunk's row.
template <typename SizeAt>
__device__ __forceinline__ int policy_bola(const EnvView& v, const SessKnobs& k, const double b, const int row,
                                           const SizeAt& size_at) {
    if (v.pol.bola_vmax <= 0.0) return 0;   // every ladder flat
    int q = 0;
    double best = 0.0;
    for (int a = 0; a < v.A; ++a) {
        const double sc = ddiv(dsub(dmul(k.bola_Vp, dadd(__ldg(v.pol.bola_v + row + a), k.bola_gp)), b), size_at(a));
        if (a == 0 || sc > best) { best = sc; q = a; }
    }
    return q;
}

// SPEC §4.6, DYNAMIC: the rule of this decision (1 = BOLA, 0 = RATE) from the one the session's last DYNAMIC decision
// left, prev, and the pre-step buffer b.  Chunk 0 ignores prev, so every episode starts on the rate rule; the strict >
// is dash.js's.
__device__ __forceinline__ int dynamic_mode(const SessKnobs& k, const int chunk, const double b, const int prev) {
    return b > (chunk != 0 && prev ? k.dyn_off : k.dyn_on) ? 1 : 0;
}

// The per-session words of a step that come straight from the SoA state (coalesced: thread i <-> session i).
struct RawState { int tr, seg, chunk, last_q; double phi, pos, buffer; };

__device__ __forceinline__ RawState load_raw(const EnvView& v, int i) {
    RawState w;
    w.tr = v.trace_id[i]; w.seg = v.seg[i]; w.chunk = v.chunk[i]; w.last_q = v.last_q[i];
    w.phi = v.phi[i]; w.pos = v.pos[i]; w.buffer = v.buffer[i];
    return w;
}

// The per-step kernel's prefetch of the NEXT tile's state words and action: asynchronous copies (cp.async, SASS LDGSTS)
// from the SoA arrays into a per-block staging buffer, every thread copying and later reading only its own session's
// words, so no barrier is involved (cp.async.wait_group makes a thread's own copies visible to it).  Prefetching into
// registers instead (the first form of this kernel) cost ten registers that do not exist under the 72-register budget
// of seven blocks per SM: ptxas spilled them, a spill store has to wait for the load it spills, and 47 % of the
// kernel's stall samples sat on those two STL instructions (ncu source page, profiles/r2z_summary.json) — the prefetch
// waited for itself.
struct NextTile {   // [kTile] columns: three doubles, five ints (the last one the action)
    double phi[kTile], pos[kTile], buffer[kTile];
    int tr[kTile], seg[kTile], chunk[kTile], last_q[kTile], action[kTile];
};

__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gmem_src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async8(void* smem_dst, const void* gmem_src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src) : "memory");
}

__device__ __forceinline__ void l2_prefetch(const void* gmem_src, const uint32_t bytes) {   // 16-byte aligned, multiple of 16
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gmem_src), "r"(bytes) : "memory");
}

// session i's words into column t of the buffer (action == nullptr: none to fetch)
__device__ __forceinline__ void request_next(NextTile& nx, const int t, const EnvView& v, const int i,
                                             const int32_t* __restrict__ action) {
    cp_async4(&nx.tr[t], v.trace_id + i); cp_async4(&nx.seg[t], v.seg + i); cp_async4(&nx.chunk[t], v.chunk + i);
    cp_async4(&nx.last_q[t], v.last_q + i);
    cp_async8(&nx.phi[t], v.phi + i); cp_async8(&nx.pos[t], v.pos + i); cp_async8(&nx.buffer[t], v.buffer + i);
    if (action) cp_async4(&nx.action[t], action + i);
}

// waits for this thread's copies and reads its column; the values are pinned in registers before the caller may
// issue the next request into the same column
__device__ __forceinline__ RawState take_next(const NextTile& nx, const int t, int& q) {
    asm volatile("cp.async.wait_all;" ::: "memory");
    RawState w;
    w.tr = nx.tr[t]; w.seg = nx.seg[t]; w.chunk = nx.chunk[t]; w.last_q = nx.last_q[t];
    w.phi = nx.phi[t]; w.pos = nx.pos[t]; w.buffer = nx.buffer[t];
    q = nx.action[t];
    asm volatile("" : "+r"(w.tr), "+r"(w.seg), "+r"(w.chunk), "+r"(w.last_q), "+d"(w.phi), "+d"(w.pos), "+d"(w.buffer), "+r"(q) :: "memory");
    return w;
}

// `m`: the trace's 32-byte record (TraceMeta), read by the caller — one 256-bit read-only load, or the block's
// shared-memory copy of it when the session follows the trace whose rows the block has staged.
__device__ __forceinline__ void make_sess(const EnvView& v, int i, const RawState& w, Sess& s, const Quad& m) {
    const int tr = w.tr;
    s.cum = v.trace_cum + (size_t)tr * cum_stride(v.T_max);
    s.idx = v.trace_idx + (size_t)tr * idx_stride(v.T_max);
    s.tab = v.tab;
    s.I = m.a; s.P = m.b; s.scale = m.c; s.T = __double2loint(m.d); s.M = __double2hiint(m.d);
    s.Td = (double)s.T;
    s.inv_I = pow2_inverse(s.I);
    s.cum_s = s.idx_s = s.tab_s = 0u;
#ifdef ABR_CHECKED
    s.chk_cum_n = cum_stride(v.T_max); s.chk_idx_n = idx_stride(v.T_max); s.chk_tab_n = v.V * v.A;
    ABR_CHECK(tr >= 0 && tr < v.n_traces, "trace id");
    ABR_CHECK(s.T >= 1 && s.T <= v.T_max && s.M >= 0 && s.M + 1 <= idx_stride(v.T_max) + (s.M == 0 ? 1 : 0), "trace record");
    ABR_CHECK(w.seg >= 0 && w.seg < s.T, "segment of the session");
#endif
    s.seg = w.seg;
    s.chunk = w.chunk;
    s.last_q = w.last_q;
    s.phi = w.phi;
    s.pos = w.pos;
    s.buffer = w.buffer;
    s.done = v.p.auto_reset ? false : (v.done[i] != 0);
    s.hist_len = v.p.track_history ? v.hist_len[i] : 0;
}

__device__ __forceinline__ void make_sess(const EnvView& v, int i, const RawState& w, Sess& s) {
    make_sess(v, i, w, s, ldg256(v.trace_meta + w.tr));
}

__device__ __forceinline__ void load_sess(const EnvView& v, int i, Sess& s) {
    const RawState w = load_raw(v, i);
    make_sess(v, i, w, s);
}

// Builds the per-trace tables of SPEC §3.1, one thread per trace (the accumulation is sequential by definition;
// runs once per environment): C[0] = 0, C[j+1] = C[j] + (bw[j]*payload)*I, and the bucket index over C (abr_common.cuh):
// cell(x) = min((int)(x * scale), M - 1) is non-decreasing in x, so with idx[b] = #{interior boundaries j in 1..T-1 :
// cell(C[j]) < b} every x of cell b satisfies C[idx[b]] <= x, and the boundaries above idx[b+1] lie beyond x.
// ok = 0 flags a trace whose period capacity is not a positive finite number or that holds a segment without capacity.
__global__ void __launch_bounds__(kStepBlock)
abr_trace_table_kernel(EnvView v, double* __restrict__ cum, uint16_t* __restrict__ idx, int32_t* __restrict__ ok_out,
                       TraceMeta* __restrict__ meta) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= v.n_traces) return;
    const double kInf = __longlong_as_double(0x7ff0000000000000ll);
    const int T = v.trace_len[t];
    const double I = v.trace_interval[t];
    const double* bw = v.trace_bw + (size_t)t * v.T_max;
    double* c_row = cum + (size_t)t * cum_stride(v.T_max);
    double c = 0.0, mincap = kInf;
    c_row[0] = 0.0;
#pragma unroll 8
    for (int j = 0; j < T; ++j) {
        const double c_next = dadd(c, dmul(dmul(bw[j], v.p.payload), I));
        c_row[j + 1] = c_next;
        mincap = fmin(mincap, dsub(c_next, c));   // the capacity the step sees: C[j+1] - C[j]
        c = c_next;
    }
    for (int j = T + 1; j < cum_stride(v.T_max); ++j) c_row[j] = kInf;
    const bool ok = c > 0.0 && c < kInf && mincap > 0.0;
    // no index rows at all when the longest trace is too long for 16-bit entries: every trace then bisects
    int M = idx_stride(v.T_max) > 0 ? idx_cells(T) : 0;
    double scale = 0.0;
    if (M > 0 && ok) {
        scale = ddiv((double)M, c);
        if (!(scale > 0.0) || !(scale < kInf)) M = 0;   // period capacity too small to scale: bisection instead
    } else {
        M = 0;
    }
    if (idx_stride(v.T_max) > 0) {
        uint16_t* i_row = idx + (size_t)t * idx_stride(v.T_max);
        int j = 1;   // next interior boundary not yet known to lie in a cell below b
        for (int b = 0; b <= M; ++b) {
            while (j <= T - 1 && (int)cell_of(c_row[j], scale, M) < b) ++j;
            i_row[b] = (uint16_t)(j - 1);
        }
        for (int b = M + 1; b < idx_stride(v.T_max); ++b) i_row[b] = (uint16_t)(T > 0 ? T - 1 : 0);
    }
    ok_out[t] = ok ? 1 : 0;
    TraceMeta m;
    m.I = I; m.P = c; m.scale = scale; m.T = T; m.M = M;
    meta[t] = m;
}

// SPEC §2 for one session: the validated trace and the position (seg, phase, data position) of the start offset.
// Shared by the reset kernel and the episode kernel's fused reset, so that both perform the same operations.
__device__ __forceinline__ void reset_seg_phase(const double I, const int T, const double off, int& seg_out,
                                                double& phi_out, int& n_bad) {
    const double x = ddiv(off, I);
    const double n = floor(x);
    // n mod T: the 32-bit remainder when n fits (every realistic offset), fmod otherwise — the same value
    int seg = (n >= 0.0 && n < 2147483648.0) ? (int)((uint32_t)n % (uint32_t)T) : (int)fmod(n, (double)T);
    double phi = dsub(x, n);   // exact, in [0, 1)
    if (seg < 0 || seg >= T) { ++n_bad; seg = 0; }
    if (!(phi >= 0.0 && phi < 1.0)) { ++n_bad; phi = 0.0; }   // NaN / infinite start offset
    seg_out = seg; phi_out = phi;
}

__device__ __forceinline__ RawState reset_position(const EnvView& v, int tr, const double off, int& n_bad) {
    RawState w;
    if (tr < 0 || tr >= v.n_traces) { ++n_bad; tr = 0; }
    const int T = v.trace_len[tr];
    const double I = v.trace_interval[tr];
    int seg;
    reset_seg_phase(I, T, off, seg, w.phi, n_bad);
    const double* c_row = v.trace_cum + (size_t)tr * cum_stride(v.T_max);
    const double c0 = __ldg(c_row + seg), c1 = __ldg(c_row + seg + 1);
    w.pos = dadd(c0, dmul(dsub(c1, c0), w.phi));
    w.tr = tr; w.seg = seg; w.chunk = 0; w.last_q = v.p.default_quality; w.buffer = 0.0;
    return w;
}

__global__ void __launch_bounds__(kStepBlock)
abr_reset_kernel(EnvView v, const int32_t* __restrict__ trace_id, const double* __restrict__ start_offset,
                 uint32_t* __restrict__ draw_counter) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= v.n) return;
    if (i == 0 && draw_counter) *draw_counter = 0u;   // SPEC §4.1: the draws of abr_env_step_policy count from the reset
    int n_bad = 0;
    const RawState w = reset_position(v, trace_id[i], start_offset ? start_offset[i] : 0.0, n_bad);
    if (n_bad) atomicAdd(v.errors, (unsigned long long)n_bad);
    v.trace_id[i] = w.tr; v.seg[i] = w.seg; v.phi[i] = w.phi; v.pos[i] = w.pos; v.buffer[i] = 0.0; v.chunk[i] = 0;
    v.last_q[i] = v.p.default_quality; v.done[i] = 0; v.hist_len[i] = 0; v.last_pred[i] = 0.0; v.err_len[i] = 0;
    v.t_now[i] = 0.0; v.play_time[i] = 0.0; v.started[i] = v.p.start_up_length <= 0.0 ? 1 : 0;
    v.play_id[i] = 0; v.play_len[i] = 0.0;
#pragma unroll
    for (int j = 0; j < ABR_NUM_ACC; ++j) v.acc[(size_t)j * v.cap + i] = 0.0;
}

// TMA bulk copy global -> shared, completion signalled on an mbarrier (byte count multiple of 16, both addresses
// 16-byte aligned).
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint32_t mbar) {
    const uint32_t dst = (uint32_t)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(gmem_src), "r"(bytes), "r"(mbar) : "memory");
}

// Wait for the given phase of an mbarrier (try_wait suspends the thread for a bounded, implementation-defined time
// per call).  The retry count is bounded so that a programming error cannot hang the GPU: a wait that gives up traps
// (the launch fails with an error the caller sees) instead of computing on whatever the buffer holds.
__device__ __forceinline__ void mbar_wait(uint32_t mbar, uint32_t parity) {
    for (int spins = 0; spins < (1 << 20); ++spins) {
        uint32_t done;
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(mbar), "r"(parity) : "memory");
        if (done) return;
    }
    __trap();
}

// Bytes of the staged copies of one trace's rows (multiples of 16): C[0..T] plus at least three of the +inf entries
// behind it (the branch-free head reads C[j0 + 1 .. j0 + 4] with j0 <= T - 1), and idx[0..M].
__device__ __forceinline__ uint32_t row_bytes_of(int T) { return (uint32_t)((T + 5) / 2) * 16u; }
__device__ __forceinline__ uint32_t idx_bytes_of(int M) { return (uint32_t)((M + 1 + 7) / 8) * 16u; }

// One chunk step of one session with the state in HBM (SPEC §3, §7).
// FAST: the five f64 outputs and end_of_video requested, no throughput history / accumulators, auto_reset on —
// compiled without the null checks and the inert/history/accumulator bookkeeping (next_sizes and throughput stay
// optional in both variants).
// OT: element type of the outputs (double, or float for the optional fp32-output mode: arithmetic stays fp64).
// SPEC §4.1: the action of a policy-in-the-loop step.  Greedy: the first arg max of the session's logits.  Sampled:
// Gumbel-max — arg max of logits[a] - ln(-ln(u_a)) is a draw from softmax(logits) — with u_a = (x_a + 0.5) / 2^23 in
// (0, 1), x_a the upper 23 bits of word a mod 4 of the Philox4x32-10 block with counter (global session index,
// draw index, a div 4) and the caller's seed as key; fp32 arithmetic.  A NaN score never wins; all-NaN gives 0.
__device__ __forceinline__ int policy_action(const EnvView& v, const StepPolicy& pol, const int i) {
    const int A = v.A;
    const float* __restrict__ row = pol.logits + (size_t)i * A;
    const bool sample = pol.draw != nullptr;
    const uint32_t draw = sample ? __ldg(pol.draw) : 0u;
    const unsigned long long g = (unsigned long long)(v.session_base + (v.perm ? __ldg(v.perm + i) : i));
    float best = __int_as_float(0xff800000);   // -inf
    int arg = 0;
    for (int a0 = 0; a0 < A; a0 += 4) {
        uint4 r = make_uint4(0u, 0u, 0u, 0u);
        if (sample) r = philox4x32_10((uint32_t)g, (uint32_t)(g >> 32), draw, (uint32_t)(a0 >> 2), pol.seed_lo, pol.seed_hi);
        const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (a0 + k < A) {
                float x = __ldg(row + a0 + k);
                if (sample) {
                    const float u = __fmul_rn(__fadd_rn((float)(w[k] >> 9), 0.5f), 1.1920928955078125e-07f);   // 2^-23
                    x = __fsub_rn(x, logf(-logf(u)));
                }
                if (x > best) { best = x; arg = a0 + k; }
            }
        }
    }
    return arg;
}

// Live-mode words of session i (SPEC §7): from the SoA state, or those of a fresh reset.  speed: the [V][N] table of
// playback speeds (the speed of content chunk k is speed[k][i]), nullable = 1.0.  LIVE = 2: the speed controller's
// stored decision instead (SPEC §7.2; a reset does not touch it, and a fresh session decides at its first piece).
template <int LIVE>
__device__ __forceinline__ void load_live(const EnvView& v, Sess& s, const int i, const double* __restrict__ speed,
                                          const bool fresh) {
    if (fresh) { s.t_now = 0.0; s.play_time = 0.0; s.play_len = 0.0; s.play_id = 0; s.started = v.p.start_up_length <= 0.0; }
    else {
        s.t_now = v.t_now[i]; s.play_time = v.play_time[i]; s.started = v.started[i] != 0;
        s.play_id = v.play_id[i]; s.play_len = v.play_len[i];
    }
    s.speed = speed ? speed + i : nullptr;
    s.speed_stride = (size_t)v.n; s.V = v.V; s.bad_speed = false;
    if constexpr (LIVE == 2) { s.play_speed = v.spd.play_speed[i]; s.ctl = &v.spd; }
}

// The SoA state words a step changes (LIVE: with the live-mode ones).
template <int LIVE>
__device__ __forceinline__ void store_state(const EnvView& v, const Sess& s, const int i) {
    v.seg[i] = s.seg; v.chunk[i] = s.chunk; v.last_q[i] = s.last_q; v.phi[i] = s.phi; v.pos[i] = s.pos;
    v.buffer[i] = s.buffer;
    if (LIVE) {
        v.t_now[i] = s.t_now; v.play_time[i] = s.play_time; v.started[i] = s.started ? 1 : 0;
        v.play_id[i] = s.play_id; v.play_len[i] = s.play_len;
    }
    if constexpr (LIVE == 2) v.spd.play_speed[i] = s.play_speed;
}

// A step's trajectory outputs at element ix of [steps][N], streamed out (st.global.cs).  FAST: the five f64 outputs and
// end_of_video are all requested and stored without null checks; NOOUT: none is requested; LIVE: the latency too,
// where requested.
template <bool FAST, bool NOOUT, int LIVE, typename OT>
__device__ __forceinline__ void store_step(const StepOutputs<OT>& o, const uint32_t ix, const StepRes& r) {
    if (NOOUT) {
    } else if (FAST) {
        __stcs(o.delay + ix, (OT)r.delay); __stcs(o.sleep + ix, (OT)r.sleep); __stcs(o.buffer + ix, (OT)r.buffer);
        __stcs(o.rebuf + ix, (OT)r.rebuf); __stcs(o.reward + ix, (OT)r.reward);
        o.eov[ix] = r.eov ? 1 : 0;
    } else {
        if (o.delay) __stcs(o.delay + ix, (OT)r.delay);
        if (o.sleep) __stcs(o.sleep + ix, (OT)r.sleep);
        if (o.buffer) __stcs(o.buffer + ix, (OT)r.buffer);
        if (o.rebuf) __stcs(o.rebuf + ix, (OT)r.rebuf);
        if (o.reward) __stcs(o.reward + ix, (OT)r.reward);
        if (o.eov) o.eov[ix] = r.eov ? 1 : 0;
        if (LIVE && o.latency) __stcs(o.latency + ix, (OT)r.latency);
    }
}

// SPEC §4.5: what a windowed observation does with its two windows.
enum WinMode { kWinZero, kWinRoll, kWinKeep };

// SPEC §4.5: column i of the windowed observation obs[3 + 2W + A][N] from a session's state (chunk, last_q, buffer,
// done).  kWinRoll: both windows move up one entry (fp32 bits copied; every load of a group of eight is issued before
// its stores, which only reach entries that are already read) and take (thr, delay) last; kWinZero: both become 0;
// kWinKeep: neither is touched.  Every other row is one fp64 operation rounded once to fp32.
__device__ __forceinline__ void write_obs_window(const EnvView& v, const StepPolicyWindow& pol, const int i, const int chunk,
                                                 const int last_q, const double buffer, const bool done, const WinMode mode,
                                                 const double thr, const double delay) {
    const int W = pol.window, A = v.A, V = v.V;
    ABR_CHECK(i >= 0 && i < v.n && W >= 1 && W <= 32 && chunk >= 0 && (chunk < V || (done && chunk == V)),
              "windowed observation column / window / chunk");
    const size_t n = (size_t)v.n;
    float* __restrict__ ob = pol.obs + i;
    const int k_prev = chunk > 0 ? chunk - 1 : 0;
    __stcs(ob, last_q < 0 ? 0.0f : (float)dmul(__ldg(v.util + (size_t)k_prev * A + last_q), pol.w_util));
    __stcs(ob + n, (float)dmul(buffer, pol.w_buffer));
    __stcs(ob + 2 * n, (float)ddiv((double)(V - chunk), (double)V));
    float* __restrict__ wt = ob + 3 * n;                 // throughput window, oldest first
    float* __restrict__ wd = ob + (size_t)(3 + W) * n;   // download-time window
    if (mode == kWinRoll) {
        for (int w0 = 0; w0 < W - 1; w0 += 8) {
            float xt[8], xd[8];
#pragma unroll
            for (int k = 0; k < 8; ++k)
                if (w0 + k < W - 1) {
                    xt[k] = __ldcs(wt + (size_t)(w0 + k + 1) * n);
                    xd[k] = __ldcs(wd + (size_t)(w0 + k + 1) * n);
                }
#pragma unroll
            for (int k = 0; k < 8; ++k)
                if (w0 + k < W - 1) {
                    __stcs(wt + (size_t)(w0 + k) * n, xt[k]);
                    __stcs(wd + (size_t)(w0 + k) * n, xd[k]);
                }
        }
        __stcs(wt + (size_t)(W - 1) * n, (float)dmul(thr, pol.w_thr));
        __stcs(wd + (size_t)(W - 1) * n, (float)dmul(delay, pol.w_delay));
    } else if (mode == kWinZero) {
        for (int w = 0; w < W; ++w) {
            __stcs(wt + (size_t)w * n, 0.0f);
            __stcs(wd + (size_t)w * n, 0.0f);
        }
    }
    float* __restrict__ os = ob + (size_t)(3 + 2 * W) * n;
    for (int a = 0; a < A; ++a)
        __stcs(os + (size_t)a * n, done ? 0.0f : (float)dmul(__ldg(v.sizes + (size_t)chunk * A + a), pol.w_size));
}

// `q`: the action, already clamped to [0, A); `lk`: the step's table reads (the caller issues them as soon as it holds
// the session's state words, next to the read of the trace record, so that the two L2 round trips overlap).
// The outputs arrive as __restrict__ parameters (of the kernel and of this function), not as StepOutputs: nvcc drops
// the qualifier on struct members, and without it the per-step kernels lose the no-alias facts their schedule is built
// on (both forms measured slower on a B200: 0.2-0.3 us of 104 per launch at 4 Mi sessions).
// POL: 0 = the action comes from the caller, 1 = from the logits with the §4.1 observation, 2 = from the logits with
// the §4.5 windowed observation.  PolicyArgs<POL>: the kernel's policy parameter (StepPolicyWindow for POL = 2).
template <int POL> struct PolicyArg { using type = StepPolicy; };
template <> struct PolicyArg<2> { using type = StepPolicyWindow; };
template <int POL> using PolicyArgs = typename PolicyArg<POL>::type;

template <bool SMEM, bool FAST, int LIVE, int POL, typename OT>
__device__ __forceinline__ void step_session(const EnvView& v, Sess& s, const int i, const int q, const Lookup& lk,
                                             const PolicyArgs<POL>& pol, const double* __restrict__ speed,
                                             OT* __restrict__ o_delay, OT* __restrict__ o_sleep, OT* __restrict__ o_buffer,
                                             OT* __restrict__ o_rebuf, OT* __restrict__ o_reward, uint8_t* __restrict__ o_eov,
                                             OT* __restrict__ o_latency, OT* __restrict__ o_thr, OT* __restrict__ o_next_sizes) {
    if (LIVE) load_live<LIVE>(v, s, i, speed, false);
    StepRes r;
    step_core<SMEM, FAST, LIVE>(v, s, q, lk, r, (!FAST && v.p.track_history) || o_thr != nullptr || (POL && pol.obs));
    if (r.walk_error || (LIVE && s.bad_speed)) atomicAdd(v.errors, 1ull);
    if (FAST) {
        store_state<false>(v, s, i);
        __stcs(o_delay + i, (OT)r.delay); __stcs(o_sleep + i, (OT)r.sleep); __stcs(o_buffer + i, (OT)r.buffer);
        __stcs(o_rebuf + i, (OT)r.rebuf); __stcs(o_reward + i, (OT)r.reward);
        o_eov[i] = r.eov ? 1 : 0;
    } else {
        if (!r.inert) {
            store_state<LIVE>(v, s, i);
            if (v.p.track_history) {
                // ring slot of this sample = (hist_len before the step) mod K; after an auto-reset hist_len is 0
                const int prev_len = r.reset_mpc ? 0 : s.hist_len - 1;
                ABR_CHECK(prev_len >= 0, "history length");
                if (!r.reset_mpc) v.bw_hist[(size_t)(prev_len % v.K) * v.cap + i] = r.thr;
                v.hist_len[i] = s.hist_len;
            }
            if (r.reset_mpc) { v.last_pred[i] = 0.0; v.err_len[i] = 0; }
            if (s.done) v.done[i] = 1;
            if (v.p.track_acc) {
                double* a = v.acc + i;
                const size_t c = v.cap;
                a[0 * c] = dadd(a[0 * c], r.reward); a[1 * c] = dadd(a[1 * c], r.rebuf); a[2 * c] = dadd(a[2 * c], r.u);
                a[3 * c] = dadd(a[3 * c], r.smooth); a[4 * c] = dadd(a[4 * c], r.sleep);
                a[5 * c] = dadd(a[5 * c], r.delay);
                a[6 * c] = dadd(a[6 * c], 1.0);
                if (r.eov) a[7 * c] = dadd(a[7 * c], 1.0);
                if (LIVE) {
                    a[8 * c] = dadd(a[8 * c], r.startup); a[9 * c] = dadd(a[9 * c], r.area);
                    a[10 * c] = dadd(a[10 * c], r.played);
                }
            }
        }
        if (o_delay) __stcs(o_delay + i, (OT)r.delay);
        if (o_sleep) __stcs(o_sleep + i, (OT)r.sleep);
        if (o_buffer) __stcs(o_buffer + i, (OT)r.buffer);
        if (o_rebuf) __stcs(o_rebuf + i, (OT)r.rebuf);
        if (o_reward) __stcs(o_reward + i, (OT)r.reward);
        if (o_eov) o_eov[i] = r.eov ? 1 : 0;
    }
    if (POL) {   // SPEC §4.1: the chosen action, the running reward and the next observation, feature-major fp32
        if (pol.action_out) pol.action_out[i] = q;
        if (pol.reward_sum) pol.reward_sum[i] = dadd(pol.reward_sum[i], r.reward);
        if constexpr (POL == 2) {   // SPEC §4.5: from the state after the step; an end of video with auto_reset restarts the windows
            write_obs_window(v, pol, i, s.chunk, s.last_q, s.buffer, !FAST && s.done,
                             r.inert ? kWinKeep : (r.reset_mpc ? kWinZero : kWinRoll), r.thr, r.delay);
        } else if (pol.obs) {
            ABR_CHECK(i >= 0 && i < v.n && (s.chunk >= 0 && (s.chunk < v.V || s.done)), "observation column / next chunk");
            float* __restrict__ ob = pol.obs + i;
            const size_t n = (size_t)v.n;
            const int A = v.A;
            __stcs(ob, (float)dmul(r.buffer, pol.s_buffer));
            __stcs(ob + n, (float)dmul(r.thr, pol.s_thr));
            __stcs(ob + 2 * n, (float)dmul(r.delay, pol.s_delay));
            __stcs(ob + 3 * n, (float)ddiv((double)q, (double)A));
            for (int a = 0; a < A; ++a)
                __stcs(ob + (size_t)(4 + a) * n,
                       (float)((!FAST && s.done) ? 0.0 : dmul(__ldg(v.sizes + s.chunk * A + a), pol.s_size)));
        }
    }
    if (o_latency) __stcs(o_latency + i, (OT)r.latency);   // 0 outside live mode
    if (o_thr) __stcs(o_thr + i, (OT)r.thr);
    if (o_next_sizes) {
        const int A = v.A;
        for (int a = 0; a < A; ++a)
            o_next_sizes[(size_t)i * A + a] = (OT)((!FAST && s.done) ? 0.0 : __ldg(v.sizes + s.chunk * A + a));
    }
}

// <= 72 registers: 7 blocks of 128 threads per SM, one wave.  A block walks a run of consecutive tiles of 128 sessions.
// When a tile starts and ends on the same trace (callers that keep sessions sorted by trace) and the trace's C and
// index rows fit in the shared-memory buffer, the block stages them with two TMA bulk copies — once, for as long as
// the following tiles stay on that trace; no barrier is needed while the rows stay — and the probes of the lanes on
// that trace are LDS.  Every other lane reads the L2-resident tables directly (one index pair + one or two sectors of C).
// POL: the actions come from the caller's logits (policy_action) instead of `action`, and the kernel also writes the
// next observation (POL = 1: SPEC §4.1; POL = 2: the windowed observation of §4.5); never with FAST or LIVE.
// LIVE: 1 = live mode with the caller's speed table, 2 = with the speed controller of SPEC §7.2.
template <bool FAST, int LIVE, int POL, typename OT>
__global__ void __launch_bounds__(kTile, (LIVE || POL) ? 4 : kTileBlocksPerSM)
abr_step_kernel(EnvView v, const int32_t* __restrict__ action, const double* __restrict__ speed,
                OT* __restrict__ o_delay, OT* __restrict__ o_sleep, OT* __restrict__ o_buffer, OT* __restrict__ o_rebuf,
                OT* __restrict__ o_reward, OT* __restrict__ o_latency, OT* __restrict__ o_next_sizes,
                uint8_t* __restrict__ o_eov, OT* __restrict__ o_thr, int smem_doubles, int tiles_per_block,
                const PolicyArgs<POL> pol) {
    extern __shared__ __align__(16) double2 s_row2[];
    __shared__ __align__(8) unsigned long long s_mbar;
    __shared__ Quad s_meta;                      // the record of the trace whose rows are staged
    const uint32_t mbar = (uint32_t)__cvta_generic_to_shared(&s_mbar);
    if (smem_doubles != 0) {
        if (threadIdx.x == 0) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(mbar));
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncthreads();
    }
    double* s_row = reinterpret_cast<double*>(s_row2);
    uint16_t* s_idx = reinterpret_cast<uint16_t*>(s_row + smem_doubles);
    uint32_t parity = 0u;                        // phase of the next staging copy (block-uniform)
    int staged = -1;                             // trace whose rows the buffer holds (block-uniform, kept per thread)
    // the state words and the action of the next tile are requested before the current tile is computed, so that
    // two tiles of loads per warp are in flight (the kernel is bound by HBM latency x occupancy otherwise); they
    // travel through shared memory, not registers (NextTile)
    __shared__ NextTile s_next;
    const bool stream_from_hbm = (long long)v.n * 121 >= kPrefetchMinBytes;   // launch-uniform
    const int warp_u = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);  // warp index, known to be warp-uniform
    const int32_t* __restrict__ act_src = POL ? nullptr : action;
    int first_next = -1, last_next = -1;
    {
        const int t0 = blockIdx.x * tiles_per_block * kTile;
        const int i0 = t0 + threadIdx.x;
        if (i0 < v.n) request_next(s_next, threadIdx.x, v, i0, act_src);
        if (t0 < v.n) { first_next = __ldg(v.trace_id + t0); last_next = __ldg(v.trace_id + min(t0 + kTile, v.n) - 1); }
    }
    for (int k = 0; k < tiles_per_block; ++k) {
        const int tile0 = (blockIdx.x * tiles_per_block + k) * kTile;
        if (tile0 >= v.n) break;                 // block-uniform
        const int i = tile0 + threadIdx.x;
        const bool valid = i < v.n;
        // traces of the first and the last session of the tile: the same words in every thread, so decisions taken
        // on them are block-uniform without a barrier.  Equal ends mean one trace for callers that keep sessions
        // sorted by trace; a lane that disagrees anyway simply takes the global path.  (Read here, ahead of this
        // iteration's loads: a later read would wait on a scoreboard it shares with them.)
        int tr_first = first_next, tr_last = last_next;
        asm volatile("" : "+r"(tr_first), "+r"(tr_last));
        int q_next = 0;
        const RawState w = take_next(s_next, threadIdx.x, q_next);   // an invalid lane reads words nobody uses
        int q_cur = POL ? (valid ? policy_action(v, pol, i) : 0) : q_next;
        if (valid && (q_cur < 0 || q_cur >= v.A)) atomicAdd(v.errors, 1ull);
        q_cur = q_cur < 0 ? 0 : (q_cur >= v.A ? v.A - 1 : q_cur);
        // The table reads depend on nothing but the state words: issued here, ahead of the staging decision and the
        // trace record (with seven blocks per SM the L1 is ~20 KB and streams state and outputs, so both are L2 round
        // trips more often than not; back to back they were 33 % of the kernel's stall samples).
        Sess s;
        Lookup lk;
        lk.size = lk.u = lk.u_prev = 0.0;
        if (valid) {
            s.tab = v.tab; s.tab_s = 0u;
#ifdef ABR_CHECKED
            s.chk_tab_n = v.V * v.A;
#endif
            lk = lookup_tables<false>(s, v.A, v.V, w.chunk, q_cur, w.last_q, v.p.smooth_prev_ladder != 0);
        }
        if (k + 1 < tiles_per_block && tile0 + kTile < v.n) {
            if (i + kTile < v.n) request_next(s_next, threadIdx.x, v, i + kTile, act_src);
#if ABR_STEP_PF_DIST > 1
            // a tile further ahead: its words are asked into L2 (one bulk prefetch per array and warp, SASS UBLKPF:
            // handled by the copy engine, not the load/store pipe), so that more than one tile of reads per block
            // is on its way from HBM — what a block keeps in flight, not the latency of one load, bounds this kernel
            // (104 us instead of 117 per 4 Mi sessions; a distance of 3 or 4 tiles: 105 / 108 us; every lane
            // prefetching its own word with prefetch.global.L2: 106.5 us; one prefetch per array and block: no gain).
            // UBLKPF takes its address from uniform registers; ptxas walks it there with an R2UR loop (one iteration:
            // lane 0 alone is active) also when it is built from a shuffled warp index — ~18 instructions per prefetch.
            {
                const int j = tile0 + ABR_STEP_PF_DIST * kTile + 32 * warp_u;
                if (stream_from_hbm && k + ABR_STEP_PF_DIST < tiles_per_block && j + 32 <= v.n && (threadIdx.x & 31) == 0) {
                    l2_prefetch(v.trace_id + j, 128); l2_prefetch(v.seg + j, 128); l2_prefetch(v.chunk + j, 128);
                    l2_prefetch(v.last_q + j, 128); l2_prefetch(v.phi + j, 256); l2_prefetch(v.pos + j, 256);
                    l2_prefetch(v.buffer + j, 256);
                    if (act_src) l2_prefetch(act_src + j, 128);
                }
            }
#endif
            first_next = __ldg(v.trace_id + tile0 + kTile);
            last_next = __ldg(v.trace_id + min(tile0 + 2 * kTile, v.n) - 1);
        }
        const int tr = valid ? w.tr : -1;
        if (smem_doubles == 0) {                 // launch-uniform: no shared-memory row buffer
            if (valid) {
                make_sess(v, i, w, s);
                step_session<false, FAST, LIVE, POL, OT>(v, s, i, q_cur, lk, pol, speed, o_delay, o_sleep, o_buffer, o_rebuf,
                                                         o_reward, o_eov, o_latency, o_thr, o_next_sizes);
            }
            continue;
        }
        if (tr_first == tr_last && tr_first != staged) {   // block-uniform: stage another trace's rows
            __syncthreads();                     // every warp is done with the rows (and the record) the buffer holds
            if (threadIdx.x == 0) {
                const Quad m0 = ldg256(v.trace_meta + tr_first);
                s_meta = m0;                     // published by the arrive below (release), seen behind mbar_wait (acquire)
                const int T0 = __double2loint(m0.d), M0 = __double2hiint(m0.d);
                const uint32_t rb = row_bytes_of(T0), ib = idx_bytes_of(M0);   // T0 <= T_max: both fit the buffer
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(rb + ib) : "memory");
                bulk_g2s(s_row, v.trace_cum + (size_t)tr_first * cum_stride(v.T_max), rb, mbar);
                bulk_g2s(s_idx, v.trace_idx + (size_t)tr_first * idx_stride(v.T_max), ib, mbar);
            }
            mbar_wait(mbar, parity);
            parity ^= 1u;
            staged = tr_first;
        }
        if (valid) {
            if (tr == staged) {
                make_sess(v, i, w, s, s_meta);
                s.cum_s = (uint32_t)__cvta_generic_to_shared(s_row);
                s.idx_s = (uint32_t)__cvta_generic_to_shared(s_idx);
#ifdef ABR_CHECKED
                s.chk_cum_n = smem_doubles; s.chk_idx_n = idx_stride(v.T_max);
                ABR_CHECK(row_bytes_of(s.T) <= 8u * (uint32_t)smem_doubles && idx_bytes_of(s.M) <= 2u * (uint32_t)idx_stride(v.T_max),
                          "staged rows fit the shared-memory buffer");
#endif
                step_session<true, FAST, LIVE, POL, OT>(v, s, i, q_cur, lk, pol, speed, o_delay, o_sleep, o_buffer, o_rebuf,
                                                        o_reward, o_eov, o_latency, o_thr, o_next_sizes);
            } else {
                make_sess(v, i, w, s);
                step_session<false, FAST, LIVE, POL, OT>(v, s, i, q_cur, lk, pol, speed, o_delay, o_sleep, o_buffer, o_rebuf,
                                                         o_reward, o_eov, o_latency, o_thr, o_next_sizes);
            }
        }
    }
}

// Per-session QoE cost of Simulator.calculate_qoe (Simulator.py:83-86) from the accumulators:
// rebuffer_weight * sum(rebuffer) + variance_weight * sum(|delta utility|), plus in live mode
// startup_weight * start-up time + latency_weight * average_latency, where the reference's average_latency is the
// sum over the playing ticks of the instantaneous latency divided by the content played (Simulator.py:179-180: the
// running mean is weighted by play_time), i.e. the latency integral per tick: area / (latency_tick * played).
__device__ __forceinline__ double session_cost(const EnvView& v, const double rebuf, const double smooth,
                                               const double played, const double startup, const double area) {
    double c = dadd(dmul(v.p.rebuf_penalty, rebuf), dmul(v.p.smooth_penalty, smooth));
    if (v.p.live) {   // + sw*start_up_time + lw*average_latency (Simulator.py:85-86)
        c = dadd(c, dmul(v.p.startup_penalty, startup));
        c = dadd(c, dmul(v.p.latency_penalty, played > 0.0 ? ddiv(area, dmul(v.p.latency_tick, played)) : 0.0));
    }
    return c;
}

// ---- SPEC §6: the statistics vector from per-block partial sums, in a fixed order and without a serial tail ----
// The block partials are cut into groups of kStatsGroup consecutive blocks.  A group's sum is formed by one block of
// (at least) 64 threads: thread (q, j) adds the eight partials 8q .. 8q+7 of the group for statistic j in ascending
// order (all eight loads issued before the first addition), then ((s0 + s1) + s2) + s3.  The final sum over the
// groups: thread (q, j) adds the group sums q, q+4, q+8, ... in ascending order, then ((s0 + s1) + s2) + s3 again.
// Who does the work does not change the order: in the fused episode the block that finishes last within a group
// reduces the group (while other groups are still running) and the group that finishes last does the final sum, so
// the tail behind the last episode is two short rounds of loads instead of a second launch; abr_stats_stage2 runs
// the same two functions with one block per group.  Missing partials count as +0.0.
constexpr int kStatsGroup = 32;
constexpr int kStatsLanes = 4 * ABR_NUM_ACC;   // threads (q, j) at work

// The "I am done" count of the statistics reduction: one acq_rel atomic by one thread of the block, behind a block
// barrier.  Release: the barrier puts the partials the block's other threads stored before this thread's atomic
// (causality order is cumulative), so whoever reads the count they led to also sees them.  Acquire: the block that
// reads the last count may — after its next block barrier — load every partial counted before (the loads bypass L1).
// __threadfence() on both sides did the same job with four MEMBAR.SC.GPU + CCTL.IVALL sequences on the chain behind
// the last episode, two of them executed by every thread of the block (each waits for its own trajectory stores).
__device__ __forceinline__ unsigned count_done(unsigned* counter) {
    unsigned old;
    asm volatile("atom.add.acq_rel.gpu.global.u32 %0, [%1], 1;" : "=r"(old) : "l"(counter) : "memory");
    return old;
}

__device__ __forceinline__ void stats_group_sum(const double* __restrict__ partials, const int n_partials, const int g,
                                                double* __restrict__ group_partials, double (*sm)[ABR_NUM_ACC]) {
    const int t = threadIdx.x;
    if (t < kStatsLanes) {
        const int q = t / ABR_NUM_ACC, j = t - q * ABR_NUM_ACC;
        const int b0 = g * kStatsGroup + q * 8;
        double x[8];
#pragma unroll
        for (int k = 0; k < 8; ++k)   // L1 is bypassed: the partials were written by other SMs
            x[k] = b0 + k < n_partials ? __ldcg(partials + (size_t)(b0 + k) * ABR_NUM_ACC + j) : 0.0;
        double s = x[0];
#pragma unroll
        for (int k = 1; k < 8; ++k) s = dadd(s, x[k]);
        sm[q][j] = s;
    }
    __syncthreads();
    if (t < ABR_NUM_ACC) group_partials[(size_t)g * ABR_NUM_ACC + t] = dadd(dadd(dadd(sm[0][t], sm[1][t]), sm[2][t]), sm[3][t]);
}

__device__ __forceinline__ void stats_final_sum(const double* __restrict__ group_partials, const int n_groups,
                                                double* __restrict__ out, double (*sm)[ABR_NUM_ACC]) {
    const int t = threadIdx.x;
    __syncthreads();   // sm may still be read by stats_group_sum's last step
    if (t < kStatsLanes) {
        const int q = t / ABR_NUM_ACC, j = t - q * ABR_NUM_ACC;
        double s = 0.0;
        for (int g0 = q; g0 < n_groups; g0 += 32) {   // eight loads in flight per thread
            double x[8];
#pragma unroll
            for (int k = 0; k < 8; ++k)
                x[k] = g0 + 4 * k < n_groups ? __ldcg(group_partials + (size_t)(g0 + 4 * k) * ABR_NUM_ACC + j) : 0.0;
#pragma unroll
            for (int k = 0; k < 8; ++k) s = dadd(s, x[k]);
        }
        sm[q][j] = s;
    }
    __syncthreads();
    if (t < ABR_NUM_ACC) out[t] = dadd(dadd(dadd(sm[0][t], sm[1][t]), sm[2][t]), sm[3][t]);
}

// Called by every thread of a block (>= 64 threads) once the block's partial `b` of `n_partials` is written (by threads
// < ABR_NUM_ACC): counts the block as finished (count_done); the last block of its group sums the
// group, the last group sums the groups into `out`.  counters[0] counts finished groups, counters[1 + g] the
// finished blocks of group g; all are left at zero.
__device__ __forceinline__ void stats_finish(const double* __restrict__ partials, const int n_partials, const int b,
                                             const StatsScratch sc, double* __restrict__ out,
                                             double (*sm)[ABR_NUM_ACC], int* s_flag) {
    const int g = b / kStatsGroup;
    const int n_groups = (n_partials + kStatsGroup - 1) / kStatsGroup;
    const int g_size = min(kStatsGroup, n_partials - g * kStatsGroup);
    ABR_CHECK(b >= 0 && b < n_partials && g_size >= 1 && blockDim.x >= kStatsLanes, "block partial / group of the statistics");
    __syncthreads();                            // the block's partial (threads < ABR_NUM_ACC) before the count
    if (threadIdx.x == 0) *s_flag = count_done(sc.counters + 1 + g) == (unsigned)(g_size - 1) ? 1 : 0;
    __syncthreads();
    if (!*s_flag) return;                       // block-uniform
    stats_group_sum(partials, n_partials, g, sc.group_partials, sm);
    __syncthreads();                            // the group's sum before its count
    if (threadIdx.x == 0) {
        sc.counters[1 + g] = 0u;
        *s_flag = count_done(sc.counters) == (unsigned)(n_groups - 1) ? 1 : 0;
    }
    __syncthreads();
    if (!*s_flag) return;
    stats_final_sum(sc.group_partials, n_groups, out, sm);
    if (threadIdx.x == 0) sc.counters[0] = 0u;
}

template <typename OT>
struct RolloutOut {
    StepOutputs<OT> traj;                    // [steps][N]
    const double* __restrict__ speed;        // live mode only: playback speed [V][N], nullable = 1.0
    // fused reset + episode + session cost (abr_env_run_host): with in_trace_id the kernel resets every session itself
    // (SPEC §2) instead of loading its state, and out_cost receives Simulator.calculate_qoe per session.  Both may
    // be device aliases of page-locked HOST memory: the inputs are then pulled and the result pushed over PCIe by
    // the kernel, overlapped with the other blocks' episodes.
    const int32_t* __restrict__ in_trace_id; // nullable
    const double* __restrict__ in_offset;    // nullable = 0.0
    double* __restrict__ out_cost;           // nullable
    // fused statistics (SPEC §6): with out_stats the kernel's own blocks add up the per-block partial sums (stats_finish
    // above) and the block that finishes last writes the statistics vector — no second launch.
    double* __restrict__ out_stats;          // nullable; may alias page-locked host memory
    StatsScratch scratch;
};

// What the fused episode adds up over one session's steps (the accumulators of SPEC §6), and whether an auto-reset
// happened (it also clears the robust-MPC predictor state).
struct EpisodeSums {
    double rew = 0.0, reb = 0.0, u = 0.0, sm = 0.0, sl = 0.0, dl = 0.0, su = 0.0, lat = 0.0, pl = 0.0;
    int steps = 0, eps = 0;
    bool reset_mpc = false;
};

// Adds one (not inert) step.  COUNT: count it and its end of episode here, note an auto-reset and record the
// throughput sample in the history ring (hist); without COUNT the caller has all of that in closed form.
template <int LIVE, bool COUNT>
__device__ __forceinline__ void add_step(EpisodeSums& a, const StepRes& r, const EnvView& v, const Sess& s, const int i,
                                         const bool hist) {
    a.rew = dadd(a.rew, r.reward); a.reb = dadd(a.reb, r.rebuf); a.u = dadd(a.u, r.u);
    a.sm = dadd(a.sm, r.smooth); a.sl = dadd(a.sl, r.sleep); a.dl = dadd(a.dl, r.delay);
    if (LIVE) { a.su = dadd(a.su, r.startup); a.lat = dadd(a.lat, r.area); a.pl = dadd(a.pl, r.played); }
    if (COUNT) {
        a.steps += 1;
        a.eps += r.eov ? 1 : 0;
        if (r.reset_mpc) a.reset_mpc = true;
        else if (hist) v.bw_hist[(size_t)((s.hist_len - 1) % v.K) * v.cap + i] = r.thr;
    }
}

// `steps` chunk steps of one session with the state in registers (SPEC §3+§4).
// FAST: the common shape — all six trajectory outputs requested, no action trace, no throughput history,
// auto_reset on — compiled without the per-output null checks and the inert/history bookkeeping.
// NOOUT (with FAST): no trajectory output at all (statistics / per-session accumulators only, e.g. abr_env_run_host).
// LIVE (never with FAST): live-streaming semantics of SPEC §7; 2 = with the speed controller of §7.2, whose decision
// for the chunk being played stays in a register for the whole call (load_live / store_state).
//
// Software pipeline (policies whose action does not depend on the state: FIXED, RANDOM; not LIVE, whose pause gate
// moves the position before every download): iteration t holds the finished head of step t and issues the head of
// step t+1 from `head(t).target + size(t+1)` next to the tail of step t, so the index / C loads of the next step
// overlap the division and the buffer / reward arithmetic of this one.  The assumption is that step t does not
// sleep; when it does (its position moved in time) the head of step t+1 is redone from the moved position.
// The action and table reads run two steps ahead for the same reason.
// UNI (with FAST, policies that run ahead): every chunk has the same utility row, so the previous step's utility is
// the next step's "previous utility" (SPEC §3.4) — carried in a register instead of looked up.
// POLICY_BITS: the policy, with kPolicySession OR-ed in for the per-session knobs of SPEC §4.7 (BBA, RATE, BOLA and
// DYNAMIC, general and live forms only), which are loaded once per call, through the session order.
template <int POLICY_BITS, bool SMEM, bool FAST, bool NOOUT, int LIVE, bool UNI, typename OT>
__device__ __forceinline__ void rollout_session(const EnvView& v, Sess& s, const int i, const uint32_t seed_lo,
                                                const uint32_t seed_hi, const int steps, const uint32_t step_base,
                                                const int32_t* __restrict__ actions_in, const RolloutOut<OT>& o,
                                                double (&acc_new)[ABR_NUM_ACC], const bool fresh) {
    constexpr int POLICY = POLICY_BITS & ~kPolicySession;
    constexpr bool SESS = (POLICY_BITS & kPolicySession) != 0;
    static_assert(!SESS || (!FAST && !NOOUT && !UNI), "per-session knobs run in the general and live forms only");
    constexpr bool AHEAD = (POLICY == ABR_POLICY_FIXED || POLICY == ABR_POLICY_RANDOM) && !LIVE;
    // the random policy is keyed by the caller's session index, whatever order the environment keeps the sessions in
    const unsigned long long gsession = (unsigned long long)(v.session_base + (v.perm ? __ldg(v.perm + i) : i));
    EpisodeSums sum;
    const int chunk_in = s.chunk;
    bool flagged = false;
    const uint32_t n = (uint32_t)v.n;
    const bool hist = !FAST && v.p.track_history != 0;
    const bool prev_ladder = v.p.smooth_prev_ladder != 0;
    uint32_t packed = 0u;   // random policy: the eight actions of one Philox block, one per nibble
    // DYNAMIC keeps the session's active rule in `packed` for the whole call and stores it back at its end.  (The
    // register is shared, and every DYNAMIC statement is an `if constexpr`, so that the other policies' forms compile
    // to the instructions they compiled to before DYNAMIC existed.)
    if constexpr (POLICY == ABR_POLICY_DYNAMIC) packed = v.pol.dyn_mode[i];
    if (LIVE) load_live<LIVE>(v, s, i, o.speed, fresh);
    SessKnobs kn;
    if constexpr (SESS) kn = session_knobs<POLICY>(v, i);
    // SPEC §4 action of step t; must be called with increasing t.  FIXED clamps t to the last row so that the
    // calls that run ahead of the final step stay inside the caller's table.
    auto action_at = [&](const int t) -> int {
        if (POLICY == ABR_POLICY_FIXED) {
            int a = __ldg(actions_in + (size_t)(t < steps ? t : steps - 1) * n + i);
            if (a < 0 || a >= v.A) { flagged = true; a = a < 0 ? 0 : v.A - 1; }
            return a;
        }
        if (POLICY == ABR_POLICY_RANDOM) {
            const uint32_t tg = step_base + (uint32_t)t;   // step index since the last reset (SPEC §4)
            if ((tg & 7u) == 0u || t == 0) {   // one Philox block per eight steps: counter = (session, step / 8),
                                               // 16-bit slice step % 8 (low half of word 0 first)
                // the key enters through an empty asm so that its ten-round schedule is recomputed here (18 additions
                // per eight steps) instead of being hoisted out of the step loop into 18 live registers
                uint32_t k_lo = seed_lo, k_hi = seed_hi;
                asm volatile("" : "+r"(k_lo), "+r"(k_hi));
                const uint4 r = philox4x32_10((uint32_t)gsession, (uint32_t)(gsession >> 32), tg >> 3, 0u,
                                              k_lo, k_hi);
                const uint32_t A = (uint32_t)v.A;   // <= 16: an action fits a nibble, (x16 * A) >> 16 < A
                auto two = [A](uint32_t x) { return (((x & 0xffffu) * A) >> 16) | ((((x >> 16) * A) >> 16) << 4); };
                packed = two(r.x) | (two(r.y) << 8) | (two(r.z) << 16) | (two(r.w) << 24);
            }
            return (int)((packed >> (4 * (tg & 7u))) & 0xfu);
        }
        // the rules' knobs: the session's, loaded once per call, or the environment-wide ones, read from the view here
        SessKnobs k;
        if constexpr (SESS) k = kn;
        else k = env_knobs(v);
        if constexpr (POLICY == ABR_POLICY_DYNAMIC) {   // only the active rule is evaluated
            if (!FAST && s.done) return 0;   // chunk == V: no sizes row (the step is inert, the rule is kept)
            const int row = s.chunk * v.A;
            ABR_CHECK(s.chunk >= 0 && s.chunk < v.V, "policy row");
            auto size_at = [&](const int a) -> double {
                return SMEM ? lds_f64(s.tab_s + 16u * (uint32_t)(row + a)) : __ldg(&s.tab[row + a].x);
            };
            packed = (uint32_t)dynamic_mode(k, s.chunk, s.buffer, (int)packed);
            return packed ? policy_bola(v, k, s.buffer, row, size_at) : policy_rate(v, k, i, s.hist_len, size_at);
        }
        if (POLICY == ABR_POLICY_RATE || POLICY == ABR_POLICY_BOLA) {
            if (!FAST && s.done) return 0;   // chunk == V: no sizes row (the step is inert)
            const int row = s.chunk * v.A;
            ABR_CHECK(s.chunk >= 0 && s.chunk < v.V, "policy row");
            // the chunk's sizes from the staged {size, utility} table or the global one
            auto size_at = [&](const int a) -> double {
                return SMEM ? lds_f64(s.tab_s + 16u * (uint32_t)(row + a)) : __ldg(&s.tab[row + a].x);
            };
            if (POLICY == ABR_POLICY_RATE) return policy_rate(v, k, i, s.hist_len, size_at);
            return policy_bola(v, k, s.buffer, row, size_at);
        }
        return policy_bba(v, k, s.buffer);
    };
    // chunk index / previous quality the step after (chunk, q) will see (SPEC §3.5), without running the step
    const int V_ = v.V, dq_ = v.p.default_quality;
    const bool wraps = FAST || v.p.auto_reset;
    auto next_chunk = [&](const int chunk) -> int {
        const int c = chunk + 1;
        return (c >= V_ && wraps) ? 0 : c;
    };
    auto next_last_q = [&](const int chunk, const int q) -> int {
        return (chunk + 1 >= V_ && wraps) ? dq_ : q;
    };
    uint32_t ix = (uint32_t)i;   // element index of (step t, session i) in the [steps][N] outputs (< 2^32, checked by the host)
    StepRes r;
    LiveGate g;
    g.buffer = 0.0; g.rebuf = g.idle = 0.0;
    g.a.startup = g.a.area = g.a.played = g.a.tc = 0.0;
    const double inv_q = pow2_inverse(v.p.sleep_quantum);   // launch-uniform
    if (AHEAD) {
        const AbrParams& pl = v.p;
        const int Vr = v.V;
        int q0 = action_at(0);
        Lookup lk0 = lookup_tables<SMEM>(s, v.A, Vr, s.chunk, q0, s.last_q, prev_ladder);
        int c1 = next_chunk(s.chunk);            // chunk index / previous quality step t+1 will see
        int lq1 = next_last_q(s.chunk, q0);
        // UNI: the utility an auto-reset leaves as "previous" (default_quality; none = no smoothness term)
        double u_dq = 0.0;
        if (UNI && dq_ >= 0) u_dq = SMEM ? lds_f64(s.tab_s + 16u * (uint32_t)dq_ + 8u) : __ldg(&s.tab[dq_].y);
        Head h;
        bool werr = false;
        head<SMEM>(s, dadd(s.pos, lk0.size), h, werr);
        const bool can_speculate = SMEM || s.M > 0;   // head_fast needs the bucket index
        bool calm = true;   // warp-uniform: no lane of the warp slept in the previous step
        const unsigned lanes = __activemask();   // the warp's sessions (converged here; all run `steps` iterations)
#pragma unroll kRolloutUnroll
        for (int t = 0; t < steps; ++t) {
            // action, table reads and head of step t+1, assuming that step t does not sleep.  Sessions whose buffer
            // sits at the cap sleep after every chunk, and the lanes of a warp tend to do so together (same trace):
            // a warp that slept in the last step does not speculate (its head would be redone anyway).
            const int q1 = action_at(t + 1);
            Lookup lk1;
            if (UNI) {
                ABR_CHECK(c1 >= 0 && c1 < Vr && q1 >= 0 && c1 * v.A + q1 < s.chk_tab_n, "{size, utility} table entry");
                const double2 su = SMEM ? lds_f64x2(s.tab_s + 16u * (uint32_t)(c1 * v.A + q1)) : __ldg(s.tab + c1 * v.A + q1);
                lk1.size = su.x;
                lk1.u = su.y;
                lk1.u_prev = c1 != 0 ? lk0.u : (dq_ >= 0 ? u_dq : su.y);   // c1 == 0: step t ends an episode
            } else {
                lk1 = lookup_tables<SMEM>(s, v.A, Vr, c1, q1, lq1, prev_ladder);
            }
            Head h1;
            bool ok1 = false;
            if (calm && can_speculate) ok1 = head_fast<SMEM>(s, dadd(h.target, lk1.size), h1);
            // tail of step t
            ABR_CHECK((unsigned long long)ix < (unsigned long long)steps * n, "trajectory element index");
            const bool moved = step_tail<SMEM, FAST, false>(pl, Vr, s, h, q0, lk0, g, r, hist, inv_q);
            store_step<FAST, NOOUT, false>(o.traj, ix, r);
            if (!FAST && o.traj.actions) __stcs(o.traj.actions + ix, q0);
            // FAST: every step counts and every V-th ends an episode (closed form below)
            if (FAST || !r.inert) add_step<false, !FAST>(sum, r, v, s, i, hist);
            calm = !__any_sync(lanes, moved);
            if (moved || !ok1) {   // s.pos: where step t left the session
                const double raw = dadd(s.pos, lk1.size);
                if (!can_speculate || !head_fast<SMEM>(s, raw, h1)) head_any<SMEM>(s, raw, h1, werr);
            }
            h = h1;
            lk0 = lk1;
            q0 = q1;
            if (!UNI) lq1 = next_last_q(c1, q1);
            c1 = next_chunk(c1);
            ix += n;
        }
        flagged |= werr;
    } else {
        for (int t = 0; t < steps; ++t) {
            const int q = action_at(t);
            const Lookup lk = lookup_tables<SMEM>(s, v.A, v.V, s.chunk, q, s.last_q, prev_ladder);
            ABR_CHECK((unsigned long long)ix < (unsigned long long)steps * n, "trajectory element index");
            step_core<SMEM, FAST, LIVE>(v, s, q, lk, r, hist);
            flagged |= r.walk_error;
            store_step<FAST, NOOUT, LIVE>(o.traj, ix, r);
            if (!FAST && o.traj.actions) __stcs(o.traj.actions + ix, q);
            if (FAST || !r.inert) add_step<LIVE, true>(sum, r, v, s, i, hist);
            ix += n;
        }
    }
    if (FAST && AHEAD) {   // auto_reset is on: the session ran `steps` steps and wrapped every V chunks
        sum.steps = steps;
        sum.eps = (int)(((long long)chunk_in + steps) / v.V);
        sum.reset_mpc = sum.eps > 0;
    }
    if (flagged || (LIVE && s.bad_speed)) atomicAdd(v.errors, 1ull);
    store_state<LIVE>(v, s, i);
    if constexpr (POLICY == ABR_POLICY_DYNAMIC) v.pol.dyn_mode[i] = (uint8_t)packed;
    if (hist) v.hist_len[i] = s.hist_len;
    if (sum.reset_mpc) { v.last_pred[i] = 0.0; v.err_len[i] = 0; }
    if (!FAST && s.done) v.done[i] = 1;
    if (fresh) {   // the rest of what abr_reset_kernel writes
        if (!hist) v.hist_len[i] = 0;
        if (!sum.reset_mpc) { v.last_pred[i] = 0.0; v.err_len[i] = 0; }
        if (FAST || !s.done) v.done[i] = 0;
        if (!LIVE) {
            v.t_now[i] = 0.0; v.play_time[i] = 0.0; v.started[i] = v.p.start_up_length <= 0.0 ? 1 : 0;
            v.play_id[i] = 0; v.play_len[i] = 0.0;
        }
    }
    // accumulator read-modify-write: all loads first (one memory round trip instead of ten dependent ones)
    double* a = v.acc + i;
    const size_t c = v.cap;
    const double add[ABR_NUM_ACC] = {sum.rew, sum.reb, sum.u, sum.sm, sum.sl, sum.dl,
                                     (double)sum.steps, (double)sum.eps,   // exact: counts below 2^31
                                     sum.su, sum.lat, sum.pl};
    double old[ABR_NUM_ACC];
#pragma unroll
    for (int j = 0; j < ABR_NUM_ACC; ++j) old[j] = fresh ? 0.0 : __ldcg(a + j * c);
#pragma unroll
    for (int j = 0; j < ABR_NUM_ACC; ++j) {
        acc_new[j] = dadd(old[j], add[j]);
        a[j * c] = acc_new[j];
    }
    if (o.out_cost) o.out_cost[i] = session_cost(v, acc_new[ABR_ACC_REBUF], acc_new[ABR_ACC_SMOOTH], acc_new[ABR_ACC_PLAY],
                                                 acc_new[ABR_ACC_STARTUP], acc_new[ABR_ACC_LATENCY]);
}

// smem_doubles: capacity of the dynamic shared-memory C-row buffer (0 disables the shared-memory path); the buffer
// is followed by the index row (idx_stride(T_max) 16-bit words, 16-byte aligned) and the sizes and utility tables.
// 8 blocks (16 warps) per SM: <= 128 registers, so that the 1 024 blocks of the 65 536-session shape are all
// co-resident (6.9 per SM).
template <int POLICY, bool FAST, bool NOOUT, int LIVE, bool UNI, typename OT>
#ifndef ABR_ROLLOUT_MINBLOCKS
#define ABR_ROLLOUT_MINBLOCKS 8   // <= 128 registers.  Registers are allocated per warp in steps of 32 per thread, so 129..160
                                  // registers mean 12 warps = six 64-thread blocks per SM (measured: 140 and 144 registers
                                  // both run 65 536 sessions in two waves, 66-69 us instead of 50) — and shared memory
                                  // (29 KB per block at the benchmark shape) allows seven, which is what one wave needs
#endif
__global__ void __launch_bounds__(kRolloutBlock, LIVE ? 6 : ABR_ROLLOUT_MINBLOCKS)
abr_rollout_kernel(EnvView v, uint32_t seed_lo, uint32_t seed_hi, int steps, uint32_t step_base,
                   const int32_t* __restrict__ actions_in, RolloutOut<OT> o, int smem_doubles,
                   double* __restrict__ block_partials) {
    extern __shared__ __align__(16) double2 s_row2[];
    __shared__ __align__(8) unsigned long long s_mbar;
    __shared__ int s_tr0, s_staged;
    __shared__ double s_part[4][ABR_NUM_ACC];   // two warps' partial sums; four rows for stats_finish
    __shared__ int s_flag;
    // let a dependent grid launched with programmatic stream serialization (the statistics stage 2) become resident
    // now; it waits for this grid's completion itself (griddepcontrol.wait), so only its launch latency is hidden
    asm volatile("griddepcontrol.launch_dependents;");
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = i < v.n;
    double acc_new[ABR_NUM_ACC];
#pragma unroll
    for (int j = 0; j < ABR_NUM_ACC; ++j) acc_new[j] = 0.0;
    Sess s;
    int tr = -1;
    const bool fresh = o.in_trace_id != nullptr;   // fused reset (launch-uniform)
    int n_bad = 0;
    // Staging (shared-memory path): the trace's C and index rows and the chunk-size / utility tables arrive by TMA bulk
    // copies (cp.async.bulk, SASS UBLKCP) that complete on an mbarrier — 29 KB per block without occupying the LSU or
    // registers.  Thread 0 issues them as soon as it knows its own trace id, i.e. one memory round trip into the
    // kernel: the whole padded rows are copied (the byte counts then depend on nothing that has to be read first),
    // and the copies run while every thread of the block is still fetching its trace record and state.  Whether the
    // block may use them (all of its sessions on that trace, and the trace has an index) is decided afterwards.
    double* s_row = reinterpret_cast<double*>(s_row2);
    uint16_t* s_idx = reinterpret_cast<uint16_t*>(s_row + smem_doubles);
    double2* s_tab = reinterpret_cast<double2*>(s_idx + idx_stride(v.T_max));
    const uint32_t mbar = (uint32_t)__cvta_generic_to_shared(&s_mbar);
    auto stage_rows = [&](const int tr0) {         // thread 0 only
        s_staged = 0;
        if (smem_doubles == 0 || tr0 < 0 || tr0 >= v.n_traces) return;
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(mbar));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        const uint32_t rb = (uint32_t)cum_stride(v.T_max) * 8u, ib = (uint32_t)idx_stride(v.T_max) * 2u;
        const uint32_t tab_bytes = (uint32_t)(v.V * v.A) * 16u;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(rb + ib + tab_bytes) : "memory");
        bulk_g2s(s_row, v.trace_cum + (size_t)tr0 * cum_stride(v.T_max), rb, mbar);
        bulk_g2s(s_idx, v.trace_idx + (size_t)tr0 * idx_stride(v.T_max), ib, mbar);
        bulk_g2s(s_tab, v.tab, tab_bytes, mbar);
        s_staged = 1;
    };
    if (valid) {
        if (fresh) {
            // SPEC §2 from the per-trace record (one dependent read after the trace id); the data position is taken
            // from the C row once it is known where that row is read from (shared memory or global)
            RawState w;
            w.tr = o.in_trace_id[i];
            if (threadIdx.x == 0) stage_rows(w.tr);
            const double off = o.in_offset ? o.in_offset[i] : 0.0;
            if (w.tr < 0 || w.tr >= v.n_traces) { ++n_bad; w.tr = 0; }
            w.seg = 0; w.chunk = 0; w.last_q = v.p.default_quality; w.phi = 0.0; w.pos = 0.0; w.buffer = 0.0;
            make_sess(v, i, w, s);
            reset_seg_phase(s.I, s.T, off, s.seg, s.phi, n_bad);
            s.done = false; s.hist_len = 0;
            tr = w.tr;
            v.trace_id[i] = tr;
            if (n_bad) atomicAdd(v.errors, (unsigned long long)n_bad);
        } else {
            tr = v.trace_id[i];
            if (threadIdx.x == 0) stage_rows(tr);
            load_sess(v, i, s);
        }
    }
    if (threadIdx.x == 0) s_tr0 = tr;            // thread 0 of a launched block is always a valid session
    __syncthreads();                              // also publishes the initialised mbarrier and s_staged
    const int tr0 = s_tr0;
    const bool staged = s_staged != 0;
    // block-uniform: the rows are there, every session of this block follows trace tr0, and tr0 has an index
    const int same = __syncthreads_and((!valid || tr == tr0) ? 1 : 0);
    const bool use_smem = staged && same && __ldg(&v.trace_meta[tr0].M) > 0;
    if (staged) mbar_wait(mbar, 0u);              // also when the rows stay unused: the copies must have landed before the block ends
    if (use_smem) {
        if (valid) {
            s.cum_s = (uint32_t)__cvta_generic_to_shared(s_row);
            s.idx_s = (uint32_t)__cvta_generic_to_shared(s_idx);
            s.tab_s = (uint32_t)__cvta_generic_to_shared(s_tab);
            // keep the addresses in registers: left alone, the compiler rematerialises them from
            // SR_CgaCtaId (an S2R round trip) at every use inside the step loop
            asm volatile("" : "+r"(s.cum_s), "+r"(s.tab_s), "+r"(s.idx_s));
#ifdef ABR_CHECKED
            s.chk_cum_n = smem_doubles; s.chk_idx_n = idx_stride(v.T_max);
            ABR_CHECK(cum_stride(v.T_max) <= smem_doubles && s.T + 4 < cum_stride(v.T_max), "staged rows fit the shared-memory buffer");
#endif
            if (fresh) s.pos = position_of<true>(s, s.seg, s.phi);
            rollout_session<POLICY, true, FAST, NOOUT, LIVE, UNI, OT>(v, s, i, seed_lo, seed_hi, steps, step_base, actions_in, o, acc_new, fresh);
        }
    } else if (valid) {
        if (fresh) s.pos = position_of<false>(s, s.seg, s.phi);
        rollout_session<POLICY, false, FAST, NOOUT, LIVE, UNI, OT>(v, s, i, seed_lo, seed_hi, steps, step_base, actions_in, o, acc_new, fresh);
    }
    // statistics stage 1 fused into the episode: per-block sums of the updated accumulators in a fixed order
    // (warp tree, then warps in ascending order), so abr_stats_partial only has to add the block partials
    if (block_partials) {
#pragma unroll
        for (int j = 0; j < ABR_NUM_ACC; ++j) {
            double x = acc_new[j];
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) x = dadd(x, __shfl_down_sync(0xffffffffu, x, d));
            if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5][j] = x;
        }
        __syncthreads();
        if (threadIdx.x < ABR_NUM_ACC) {
            double x = s_part[0][threadIdx.x];
            for (int w = 1; w < kRolloutBlock / 32; ++w) x = dadd(x, s_part[w][threadIdx.x]);
            block_partials[(size_t)blockIdx.x * ABR_NUM_ACC + threadIdx.x] = x;
        }
        if (o.out_stats) {   // launch-uniform
            static_assert(kRolloutBlock >= kStatsLanes, "stats_finish needs 44 threads");
            stats_finish(block_partials, (int)gridDim.x, (int)blockIdx.x, o.scratch, o.out_stats, s_part, &s_flag);
        }
    }
}

// ---- statistics: deterministic two-stage reduction of acc[ABR_NUM_ACC][n] (SPEC §6) ----
__device__ __forceinline__ double block_sum(double x, double* sm) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x = dadd(x, __shfl_down_sync(0xffffffffu, x, o));
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) sm[w] = x;
    __syncthreads();
    if (w == 0) {
        x = (l < (int)(blockDim.x >> 5)) ? sm[l] : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) x = dadd(x, __shfl_down_sync(0xffffffffu, x, o));
    }
    return x;  // valid in thread 0
}

__global__ void __launch_bounds__(kStatsBlock)
abr_stats_stage1(EnvView v, double* __restrict__ partials) {
    __shared__ double sm[32];
    const int lo = blockIdx.x * kStatsSessionsPerBlock;
    const int hi = min(v.n, lo + kStatsSessionsPerBlock);
    // all rows' loads are issued before any reduction so that one block keeps 8 x 4 loads per thread in flight
    double x[ABR_NUM_ACC];
#pragma unroll
    for (int j = 0; j < ABR_NUM_ACC; ++j) {
        x[j] = 0.0;
        for (int i = lo + threadIdx.x; i < hi; i += blockDim.x) x[j] = dadd(x[j], v.acc[(size_t)j * v.cap + i]);
    }
#pragma unroll
    for (int j = 0; j < ABR_NUM_ACC; ++j) {
        const double t = block_sum(x[j], sm);
        if (threadIdx.x == 0) partials[(size_t)blockIdx.x * ABR_NUM_ACC + j] = t;
    }
}

// one block per group of partials; the order of the additions is that of stats_finish, whoever runs it
__global__ void __launch_bounds__(64)
abr_stats_stage2(const double* __restrict__ partials, int n_partials, StatsScratch sc, double* __restrict__ out) {
    __shared__ double sm[4][ABR_NUM_ACC];
    __shared__ int s_flag;
    // launched with programmatic stream serialization: the grid may be resident before the kernel in front of it
    // in the stream (the episode) has finished; wait here for its completion and its writes
    asm volatile("griddepcontrol.wait;" ::: "memory");
    const int g = blockIdx.x;
    const int n_groups = (n_partials + kStatsGroup - 1) / kStatsGroup;
    stats_group_sum(partials, n_partials, g, sc.group_partials, sm);
    __syncthreads();
    if (threadIdx.x == 0) s_flag = count_done(sc.counters) == (unsigned)(n_groups - 1) ? 1 : 0;
    __syncthreads();
    if (!s_flag) return;
    stats_final_sum(sc.group_partials, n_groups, out, sm);
    if (threadIdx.x == 0) sc.counters[0] = 0u;
}

__global__ void __launch_bounds__(kStepBlock)
abr_qoe_cost_kernel(EnvView v, double* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= v.n) return;
    const size_t c = v.cap;
    out[i] = session_cost(v, v.acc[ABR_ACC_REBUF * c + i], v.acc[ABR_ACC_SMOOTH * c + i], v.acc[ABR_ACC_PLAY * c + i],
                          v.acc[ABR_ACC_STARTUP * c + i], v.acc[ABR_ACC_LATENCY * c + i]);
}

// abr_env_policy_decide: one thread per session, the same policy functions as the fused episode's action_at, on the
// state the next step starts from (in live mode the buffer before the pause gate, as in the episode).  POLICY_BITS: the
// policy, with kPolicySession OR-ed in for the per-session knobs of SPEC §4.7 (each thread reads only the fields its
// policy uses).
template <int POLICY_BITS>
__global__ void __launch_bounds__(kStepBlock)
abr_policy_decide_kernel(EnvView v, int32_t* __restrict__ action) {
    constexpr int POLICY = POLICY_BITS & ~kPolicySession;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= v.n) return;
    const double b = v.buffer[i];
    SessKnobs k;
    if constexpr ((POLICY_BITS & kPolicySession) != 0) k = session_knobs<POLICY>(v, i);
    else k = env_knobs(v);
    int q;
    if (POLICY == ABR_POLICY_BBA) {
        q = policy_bba(v, k, b);
    } else if (!v.p.auto_reset && v.done[i]) {
        q = 0;   // chunk == V: no sizes row
    } else {
        const int chunk = v.chunk[i];
        ABR_CHECK(chunk >= 0 && chunk < v.V, "policy row");
        const int row = chunk * v.A;
        auto size_at = [&](const int a) -> double { return __ldg(v.sizes + row + a); };
        if constexpr (POLICY == ABR_POLICY_DYNAMIC) {
            const int m = dynamic_mode(k, chunk, b, v.pol.dyn_mode[i]);
            v.pol.dyn_mode[i] = (uint8_t)m;
            q = m ? policy_bola(v, k, b, row, size_at) : policy_rate(v, k, i, v.hist_len[i], size_at);
        } else {
            q = POLICY == ABR_POLICY_RATE ? policy_rate(v, k, i, v.hist_len[i], size_at) : policy_bola(v, k, b, row, size_at);
        }
    }
    action[i] = q;
}

// ---- SPEC §4.4: clairvoyant lookahead (abr_env_lookahead_decide) ----
// One thread per (session, first action a0); the A threads of a session sit in consecutive lanes of one warp
// (32 / A sessions per warp, the remaining lanes idle).  A thread walks the A^(h-1) completions of its a0 depth first
// in C order, stepping a register copy of the session with the per-step kernel's own step_core; the states before
// steps 1 .. h-1 and the partial sums wait on a per-thread stack, so every node of the tree is stepped once.  The
// lane of a0 = 0 then scans the A lane results in a0 order with the same strict > as each lane's own scan, which is
// the first maximum of SPEC §4.4 over the whole tree.
constexpr int kLookaheadBlock = 128;
constexpr int kLookaheadMaxH = 8;

struct LookNode { double phi, pos, buffer, J; int seg; };   // a session's state before a step, and the sum so far

// FAST: auto_reset is on, so that no session is inert (the step drops the done bookkeeping)
template <bool FAST>
__global__ void __launch_bounds__(kLookaheadBlock)
abr_lookahead_kernel(EnvView v, const int H, int32_t* __restrict__ action, double* __restrict__ best_value,
                     int32_t* __restrict__ best_seq) {
    __shared__ double s_val[kLookaheadBlock];
    __shared__ int s_leaf[kLookaheadBlock];
    __shared__ int s_err[kLookaheadBlock];
    const int A = v.A;
    const int per_warp = 32 / A;
    const int lane = threadIdx.x & 31;
    const int g = lane / A, a0 = lane - g * A;
    const int i = (int)((blockIdx.x * (kLookaheadBlock / 32) + (threadIdx.x >> 5)) * per_warp) + g;
    const bool active = g < per_warp && i < v.n;
    double best = 0.0;
    int best_leaf = 0, h = 0, n_leaves = 1;
    bool err = false;
    if (active) {
        Sess s;
        load_sess(v, i, s);
        h = s.done ? 0 : min(H, v.V - s.chunk);
        ABR_CHECK(h <= kLookaheadMaxH && s.chunk >= 0, "lookahead depth");
        for (int d = 1; d < h; ++d) n_leaves *= A;
        if (h > 0) {
            const bool prev_ladder = v.p.smooth_prev_ladder != 0;
            const int chunk0 = s.chunk, hist0 = s.hist_len;
            LookNode st[kLookaheadMaxH];   // st[d]: the state before step d (d >= 1)
            int dig[kLookaheadMaxH];       // the sequence of the current leaf
            dig[0] = a0;
            for (int d = 1; d < h; ++d) dig[d] = 0;
            int k = 0, leaf = 0;
            double J = 0.0;
            for (;;) {
                for (int d = k; d < h; ++d) {
                    const int q = dig[d];
                    const Lookup lk = lookup_tables<false>(s, A, v.V, s.chunk, q, s.last_q, prev_ladder);
                    StepRes r;
                    step_core<false, FAST, false>(v, s, q, lk, r, false);
                    err |= r.walk_error;
                    J = dadd(J, r.reward);
                    if (d + 1 < h) {
                        LookNode& nd = st[d + 1];
                        nd.phi = s.phi; nd.pos = s.pos; nd.buffer = s.buffer; nd.J = J; nd.seg = s.seg;
                    }
                }
                if (leaf == 0 || J > best) { best = J; best_leaf = leaf; }
                int d = h - 1;   // the next leaf in C order: the deepest digit that can still grow
                while (d >= 1 && dig[d] == A - 1) dig[d--] = 0;
                if (d < 1) break;
                ++dig[d];
                ++leaf;
                k = d;
                const LookNode& nd = st[k];
                s.phi = nd.phi; s.pos = nd.pos; s.buffer = nd.buffer; J = nd.J; s.seg = nd.seg;
                s.chunk = chunk0 + k; s.last_q = dig[k - 1]; s.hist_len = hist0 + k; s.done = false;
            }
        }
    }
    s_val[threadIdx.x] = best;
    s_leaf[threadIdx.x] = a0 * n_leaves + best_leaf;
    s_err[threadIdx.x] = err ? 1 : 0;
    __syncwarp();
    if (!active || a0 != 0) return;
    int idx = s_leaf[threadIdx.x], flagged = s_err[threadIdx.x];
    for (int a = 1; a < A; ++a) {
        const double x = s_val[threadIdx.x + a];
        if (x > best) { best = x; idx = s_leaf[threadIdx.x + a]; }
        flagged |= s_err[threadIdx.x + a];
    }
    if (flagged) atomicAdd(v.errors, 1ull);
    if (h == 0) best = 0.0;
    action[i] = h > 0 ? idx / n_leaves : 0;
    if (best_value) best_value[i] = best;
    if (best_seq) {
        int32_t* row = best_seq + (size_t)i * H;
        for (int d = H - 1; d >= h; --d) row[d] = -1;
        for (int d = h - 1; d >= 0; --d) { row[d] = idx % A; idx /= A; }
    }
}

}  // namespace

// abr_shared.cu compiles everything above (the step functions its kernel is built from) and none of what follows.
#ifndef ABR_STEP_DEVICE_ONLY

cudaError_t launch_lookahead(const EnvView& v, int H, int32_t* d_action, double* d_best_value, int32_t* d_best_seq,
                             cudaStream_t st) {
    if (v.n == 0) return cudaSuccess;
    if (H < 1 || H > kLookaheadMaxH || v.A < 1 || v.A > 32) return cudaErrorInvalidValue;
    const int per_block = (kLookaheadBlock / 32) * (32 / v.A);
    const unsigned grid = (unsigned)((v.n + per_block - 1) / per_block);
    if (v.p.auto_reset) abr_lookahead_kernel<true><<<grid, kLookaheadBlock, 0, st>>>(v, H, d_action, d_best_value, d_best_seq);
    else abr_lookahead_kernel<false><<<grid, kLookaheadBlock, 0, st>>>(v, H, d_action, d_best_value, d_best_seq);
    count_launch();
    return cudaGetLastError();
}

// The decision kernel of policy P: its per-session form (SPEC §4.7) while the per-session knobs are installed.
template <int P>
static void launch_decide_form(const EnvView& v, int32_t* d_action, cudaStream_t st) {
    const unsigned grid = (v.n + kStepBlock - 1) / kStepBlock;
    if (v.sp.on) abr_policy_decide_kernel<P | kPolicySession><<<grid, kStepBlock, 0, st>>>(v, d_action);
    else abr_policy_decide_kernel<P><<<grid, kStepBlock, 0, st>>>(v, d_action);
}

cudaError_t launch_policy_decide(const EnvView& v, int policy, int32_t* d_action, cudaStream_t st) {
    if (v.n == 0) return cudaSuccess;
    switch (policy) {
        case ABR_POLICY_BBA: launch_decide_form<ABR_POLICY_BBA>(v, d_action, st); break;
        case ABR_POLICY_RATE: launch_decide_form<ABR_POLICY_RATE>(v, d_action, st); break;
        case ABR_POLICY_BOLA: launch_decide_form<ABR_POLICY_BOLA>(v, d_action, st); break;
        case ABR_POLICY_DYNAMIC: launch_decide_form<ABR_POLICY_DYNAMIC>(v, d_action, st); break;
        default: return cudaErrorInvalidValue;
    }
    count_launch();
    return cudaGetLastError();
}

// SPEC §4.7: one thread per session.  The first field that fails the check the environment-wide setters apply (in the
// field order), as 8 * session + field, into the minimum at *first; or, without `first`, the session's column of the
// table with BOLA's (Vp, gp) derived as install_policy_params derives them (fp64, no FMA).
__global__ void __launch_bounds__(kStepBlock)
abr_session_params_kernel(const SessionParamsSrc a, int n, int cap, double* __restrict__ tab,
                          unsigned long long* __restrict__ first) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n) return;
    double x[7];
#pragma unroll
    for (int f = 0; f < 7; ++f) x[f] = a.src[f] ? a.src[f][c] : a.env_wide[f];
    if (first) {
        int bad = -1;
        if (!isfinite(x[kSpBbaReservoir])) bad = kSpBbaReservoir;
        else if (!isfinite(x[kSpBbaCushion]) || !(x[kSpBbaCushion] > 0.0)) bad = kSpBbaCushion;
        else if (!isfinite(x[kSpRbSafety]) || !(x[kSpRbSafety] > 0.0)) bad = kSpRbSafety;
        else if (!isfinite(x[kSpBolaMin]) || !(x[kSpBolaMin] > 0.0)) bad = kSpBolaMin;
        else if (!isfinite(x[kSpBolaTarget]) || !(x[kSpBolaMin] < x[kSpBolaTarget])) bad = kSpBolaTarget;
        else if (!isfinite(x[kSpSwitchOn])) bad = kSpSwitchOn;
        else if (!isfinite(x[kSpSwitchOff]) || !(x[kSpSwitchOff] >= 0.0) || !(x[kSpSwitchOff] < x[kSpSwitchOn]))
            bad = kSpSwitchOff;
        if (bad >= 0) atomicMin(first, 8ull * (unsigned long long)c + (unsigned long long)bad);
        return;
    }
#pragma unroll
    for (int f = 0; f < 7; ++f) tab[(size_t)f * cap + c] = x[f];
    const double gp = ddiv(a.bola_vmax, dsub(ddiv(x[kSpBolaTarget], x[kSpBolaMin]), 1.0));
    tab[(size_t)kSpBolaGp * cap + c] = gp;
    tab[(size_t)kSpBolaVp * cap + c] = ddiv(x[kSpBolaMin], gp);
}

cudaError_t launch_session_params(const SessionParamsSrc& a, int n, int cap, double* d_tab,
                                  unsigned long long* d_first, cudaStream_t st) {
    if (d_first) {
        cudaError_t e = cudaMemsetAsync(d_first, 0xff, sizeof(unsigned long long), st);
        if (e != cudaSuccess) return e;
    }
    abr_session_params_kernel<<<(n + kStepBlock - 1) / kStepBlock, kStepBlock, 0, st>>>(a, n, cap, d_tab, d_first);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_trace_table(const EnvView& v, double* d_cum, uint16_t* d_idx, int32_t* d_ok, TraceMeta* d_meta,
                               cudaStream_t st) {
    abr_trace_table_kernel<<<(v.n_traces + kStepBlock - 1) / kStepBlock, kStepBlock, 0, st>>>(v, d_cum, d_idx, d_ok, d_meta);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_reset(const EnvView& v, const int32_t* d_trace_id, const double* d_start_offset,
                         uint32_t* d_draw_counter, cudaStream_t st) {
    if (v.n == 0) return cudaSuccess;
    abr_reset_kernel<<<(v.n + kStepBlock - 1) / kStepBlock, kStepBlock, 0, st>>>(v, d_trace_id, d_start_offset, d_draw_counter);
    count_launch();
    return cudaGetLastError();
}

// Dynamic shared memory above 48 KB needs an opt-in per kernel; long traces (up to ~18 000 segments in the fused
// kernel) then still run on the shared-memory path, with fewer blocks per SM.
constexpr size_t kSmemOptInLimit = 200 * 1024;

template <typename Kernel>
static cudaError_t allow_smem(Kernel kernel, size_t bytes) {
    if (bytes <= 48 * 1024) return cudaSuccess;
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

template <typename OT>
cudaError_t launch_step(const EnvView& v, const int32_t* d_action, const double* d_speed, const StepOutputs<OT>& o,
                        cudaStream_t st, const StepPolicyWindow* policy) {
    if (v.n == 0) return cudaSuccess;
    const bool live = v.p.live != 0;
    const StepPolicyWindow pol = policy ? *policy : StepPolicyWindow{};
    const bool fast = !policy && !live && o.has_core() && v.p.track_history == 0 && v.p.track_acc == 0 &&
                      v.p.auto_reset != 0;
    // persistent-style grid: one wave of kTileBlocksPerSM blocks per SM, each walking an equal run of consecutive
    // tiles (at least kStepTiles, so that small batches still amortise the staging); no tail wave
    static int sm_count = 0;
    if (sm_count == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
            sm_count = 148;
    }
    const int total_tiles = (v.n + kTile - 1) / kTile;
    int tiles_per_block = (total_tiles + sm_count * kTileBlocksPerSM - 1) / (sm_count * kTileBlocksPerSM);
    if (tiles_per_block < kStepTiles) tiles_per_block = kStepTiles;
    const unsigned grid = (total_tiles + tiles_per_block - 1) / tiles_per_block;
    // shared-memory buffer (C row + index row) for blocks whose sessions share a trace
    int smem_doubles = cum_smem_doubles(v.T_max);
    size_t smem_bytes = (size_t)smem_doubles * sizeof(double) + (size_t)idx_stride(v.T_max) * sizeof(uint16_t);
    if (smem_bytes > kSmemOptInLimit || idx_stride(v.T_max) == 0) { smem_doubles = 0; smem_bytes = 0; }
    auto go = [&](auto kernel) {
        cudaError_t e = allow_smem(kernel, smem_bytes);
        if (e == cudaSuccess)
            kernel<<<grid, kTile, smem_bytes, st>>>(v, d_action, d_speed, o.delay, o.sleep, o.buffer, o.rebuf, o.reward,
                                                    o.latency, o.next_sizes, o.eov, o.thr, smem_doubles, tiles_per_block, pol);
        return e;
    };
    cudaError_t e;
    if (policy) {
        if constexpr (std::is_same<OT, double>::value)
            e = pol.window > 0 ? go(abr_step_kernel<false, false, 2, OT>) : go(abr_step_kernel<false, false, 1, OT>);
        else return cudaErrorInvalidValue;
    }
    else if (live && v.spd.on) e = go(abr_step_kernel<false, 2, 0, OT>);
    else if (live) e = go(abr_step_kernel<false, true, 0, OT>);
    else if (fast) e = go(abr_step_kernel<true, false, 0, OT>);
    else e = go(abr_step_kernel<false, false, 0, OT>);
    if (e != cudaSuccess) return e;
    count_launch();
    return cudaGetLastError();
}

template cudaError_t launch_step<double>(const EnvView&, const int32_t*, const double*, const StepOutputs<double>&,
                                         cudaStream_t, const StepPolicyWindow*);
template cudaError_t launch_step<float>(const EnvView&, const int32_t*, const double*, const StepOutputs<float>&,
                                        cudaStream_t, const StepPolicyWindow*);

__global__ void abr_bump_kernel(uint32_t* counter) { *counter += 1u; }

// SPEC §4.1: the step with the action drawn from the caller's logits and the observation written by the same kernel;
// the draw counter is advanced behind it (same stream: every thread has read it by then), so that a captured graph
// replays with a new draw every time.
cudaError_t launch_step_policy(const EnvView& v, const StepPolicyWindow& pol, const StepOutputs<double>& o,
                               uint32_t* d_draw_counter, cudaStream_t st) {
    if (v.n == 0) return cudaSuccess;
    cudaError_t e = launch_step<double>(v, nullptr, nullptr, o, st, &pol);
    if (e != cudaSuccess) return e;
    if (pol.draw) {
        abr_bump_kernel<<<1, 1, 0, st>>>(d_draw_counter);
        count_launch();
    }
    return cudaGetLastError();
}

// SPEC §4.5: the windowed observation of every session's state, both windows 0 (the first observation of an episode).
__global__ void __launch_bounds__(kStepBlock) abr_observe_window_kernel(EnvView v, const StepPolicyWindow pol) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= v.n) return;
    const bool done = !v.p.auto_reset && v.done[i] != 0;
    write_obs_window(v, pol, i, v.chunk[i], v.last_q[i], v.buffer[i], done, kWinZero, 0.0, 0.0);
}

cudaError_t launch_observe_window(const EnvView& v, const StepPolicyWindow& pol, cudaStream_t st) {
    if (v.n == 0) return cudaSuccess;
    abr_observe_window_kernel<<<(v.n + kStepBlock - 1) / kStepBlock, kStepBlock, 0, st>>>(v, pol);
    count_launch();
    return cudaGetLastError();
}

// The episode kernel's compile-time form for policy P, launched by go(kernel, outputs).  The carried-utility form
// (UNI) only exists where it pays: the run-ahead loop (not the buffer-based policy).  NOOUT stores no trajectory, so
// its output type is never used: the double form serves the fp32 calls too.  live: 0 = VoD, 1 = live mode with a
// speed table, 2 = with the speed controller of SPEC §7.2.
template <int P, typename OT, typename Go>
static cudaError_t launch_rollout_form(const Go& go, const RolloutOut<OT>& o, const RolloutOut<double>& o_none,
                                       const int live, const bool fast, const bool none, const bool uni) {
    constexpr bool kAhead = P == ABR_POLICY_FIXED || P == ABR_POLICY_RANDOM;
    if (live == 2) return go(abr_rollout_kernel<P, false, false, 2, false, OT>, o);
    if (live) return go(abr_rollout_kernel<P, false, false, true, false, OT>, o);
    // RATE and DYNAMIC read the history ring: track_history = 1, never a FAST / NOOUT form
    if constexpr (P == ABR_POLICY_RATE || P == ABR_POLICY_DYNAMIC) {
        if (fast || none) return cudaErrorInvalidValue;
        return go(abr_rollout_kernel<P, false, false, false, false, OT>, o);
    } else {
        if (fast && uni) return go(abr_rollout_kernel<P, true, false, false, kAhead, OT>, o);
        if (fast) return go(abr_rollout_kernel<P, true, false, false, false, OT>, o);
        if (none && uni) return go(abr_rollout_kernel<P, true, true, false, kAhead, double>, o_none);
        if (none) return go(abr_rollout_kernel<P, true, true, false, false, double>, o_none);
        return go(abr_rollout_kernel<P, false, false, false, false, OT>, o);
    }
}

// The episode kernel's per-session form (SPEC §4.7) of a policy that reads the knobs: the general form, also where the
// environment-wide knobs would take a FAST / NOOUT form (its outputs may be null), or the live form.
template <int P, typename OT, typename Go>
static cudaError_t launch_rollout_session_form(const Go& go, const RolloutOut<OT>& o, const int live) {
    constexpr int PS = P | kPolicySession;
    if (live == 2) return go(abr_rollout_kernel<PS, false, false, 2, false, OT>, o);
    if (live == 1) return go(abr_rollout_kernel<PS, false, false, 1, false, OT>, o);
    return go(abr_rollout_kernel<PS, false, false, 0, false, OT>, o);
}

template <typename OT>
cudaError_t launch_rollout(const EnvView& v, int policy, uint64_t seed, int steps, uint32_t step_base,
                           const int32_t* d_actions_in, const double* d_speed, const StepOutputs<OT>& out,
                           double* d_block_partials, const RolloutFused& f, cudaStream_t st) {
    if (v.n == 0 || steps <= 0) return cudaSuccess;
    const dim3 grid((v.n + kRolloutBlock - 1) / kRolloutBlock), block(kRolloutBlock);
    const uint32_t lo = (uint32_t)seed, hi = (uint32_t)(seed >> 32);
    double* out_stats = d_block_partials ? f.out_stats : nullptr;
    const RolloutOut<OT> o{out, d_speed, f.in_trace_id, f.in_offset, f.out_cost, out_stats, f.scratch};
    const RolloutOut<double> o_none{StepOutputs<double>{}, d_speed, f.in_trace_id, f.in_offset, f.out_cost, out_stats, f.scratch};
    const int live = v.p.live == 0 ? 0 : (v.spd.on ? 2 : 1);
    // shared-memory buffer: the longest C row, the longest index row and the two tables
    int smem_doubles = cum_smem_doubles(v.T_max);
    size_t smem_bytes = ((size_t)smem_doubles + 2 * (size_t)v.V * v.A) * sizeof(double) +
                        (size_t)idx_stride(v.T_max) * sizeof(uint16_t);
    // <= 31 KB keeps 7 blocks per SM resident (the 65 536-session shape is then one wave); longer traces opt in to
    // more shared memory and run with fewer blocks per SM, which still beats scattered global probes
    if (smem_bytes > kSmemOptInLimit || idx_stride(v.T_max) == 0) { smem_doubles = 0; smem_bytes = 0; }
    const bool plain = !live && v.p.track_history == 0 && v.p.auto_reset != 0;
    const bool fast = plain && out.has_core() && !out.actions;
    const bool none = plain && out.none();
    const bool uni = v.uniform_util != 0;
    auto go = [&](auto kernel, const auto& o_k) {
        cudaError_t e = allow_smem(kernel, smem_bytes);
        if (e == cudaSuccess)
            kernel<<<grid, block, smem_bytes, st>>>(v, lo, hi, steps, step_base, d_actions_in, o_k, smem_doubles, d_block_partials);
        return e;
    };
    cudaError_t e;
    if (v.sp.on && policy == ABR_POLICY_BBA) e = launch_rollout_session_form<ABR_POLICY_BBA>(go, o, live);
    else if (v.sp.on && policy == ABR_POLICY_RATE) e = launch_rollout_session_form<ABR_POLICY_RATE>(go, o, live);
    else if (v.sp.on && policy == ABR_POLICY_BOLA) e = launch_rollout_session_form<ABR_POLICY_BOLA>(go, o, live);
    else if (v.sp.on && policy == ABR_POLICY_DYNAMIC) e = launch_rollout_session_form<ABR_POLICY_DYNAMIC>(go, o, live);
    else switch (policy) {
        case ABR_POLICY_FIXED: e = launch_rollout_form<ABR_POLICY_FIXED>(go, o, o_none, live, fast, none, uni); break;
        case ABR_POLICY_RANDOM: e = launch_rollout_form<ABR_POLICY_RANDOM>(go, o, o_none, live, fast, none, uni); break;
        case ABR_POLICY_BBA: e = launch_rollout_form<ABR_POLICY_BBA>(go, o, o_none, live, fast, none, uni); break;
        case ABR_POLICY_RATE: e = launch_rollout_form<ABR_POLICY_RATE>(go, o, o_none, live, fast, none, uni); break;
        case ABR_POLICY_BOLA: e = launch_rollout_form<ABR_POLICY_BOLA>(go, o, o_none, live, fast, none, uni); break;
        case ABR_POLICY_DYNAMIC:
            e = launch_rollout_form<ABR_POLICY_DYNAMIC>(go, o, o_none, live, fast, none, uni);
            break;
        default: return cudaErrorInvalidValue;
    }
    if (e != cudaSuccess) return e;
    count_launch();
    return cudaGetLastError();
}

template cudaError_t launch_rollout<double>(const EnvView&, int, uint64_t, int, uint32_t, const int32_t*, const double*,
                                            const StepOutputs<double>&, double*, const RolloutFused&, cudaStream_t);
template cudaError_t launch_rollout<float>(const EnvView&, int, uint64_t, int, uint32_t, const int32_t*, const double*,
                                           const StepOutputs<float>&, double*, const RolloutFused&, cudaStream_t);

int stats_num_partials(int n) { return n <= 0 ? 1 : (n + kStatsSessionsPerBlock - 1) / kStatsSessionsPerBlock; }

cudaError_t launch_qoe_cost(const EnvView& v, double* d_out, cudaStream_t st) {
    if (v.n == 0) return cudaSuccess;
    abr_qoe_cost_kernel<<<(v.n + kStepBlock - 1) / kStepBlock, kStepBlock, 0, st>>>(v, d_out);
    count_launch();
    return cudaGetLastError();
}

int rollout_num_blocks(int n) { return n <= 0 ? 1 : (n + kRolloutBlock - 1) / kRolloutBlock; }

// have_partials: d_partials already holds n_partials block sums (written by the fused episode kernel)
int stats_num_groups(int n_partials) { return n_partials <= 0 ? 1 : (n_partials + kStatsGroup - 1) / kStatsGroup; }

cudaError_t launch_stats(const EnvView& v, double* d_partials, int n_partials, bool have_partials, double* d_out,
                         const StatsScratch& scratch, cudaStream_t st) {
    if (v.n == 0) return cudaMemsetAsync(d_out, 0, sizeof(double) * ABR_NUM_STATS, st);   // empty batch
    if (!have_partials) {
        abr_stats_stage1<<<n_partials, kStatsBlock, 0, st>>>(v, d_partials);
        count_launch();
    }
    {   // programmatic dependent launch: scheduled while the episode kernel still runs, starts working when it is done
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(stats_num_groups(n_partials));
        cfg.blockDim = dim3(64);
        cfg.dynamicSmemBytes = 0;
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        const double* partials_c = d_partials;
        cudaError_t e = cudaLaunchKernelEx(&cfg, abr_stats_stage2, partials_c, n_partials, scratch, d_out);
        if (e != cudaSuccess) return e;
    }
    count_launch();
    return cudaGetLastError();
}

#endif  // ABR_STEP_DEVICE_ONLY

}  // namespace abr
