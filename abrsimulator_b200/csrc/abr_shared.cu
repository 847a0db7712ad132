// Shared bottleneck links (SPEC.md §9): G players share one trace's capacity equally while their downloads overlap
// (processor sharing), simulated event by event.  One warp per link, one lane per player.
//
// Every lane holds the link's position (seg, phi, pos in its Sess, the whole periods and the clock) and computes the
// same values from the same inputs, so the event loop is warp-uniform: the number of active downloads is a ballot,
// the smallest remaining download and the smallest wait are shuffle minima (exact), and the head of SPEC §3.1 — where
// the next completion would leave the link — is searched once per event by all lanes together (the same addresses: a
// broadcast).  Only the per-player work diverges: the decision at a request (lanes of different policies take turns)
// and the §3.2-§3.5 bookkeeping at a completion.
//
// Trace access: the link's C row and bucket index staged in shared memory per warp (with the {size, utility} table
// per block) when they fit, the global read-only path otherwise; the choice is launch-uniform (launch_shared).
//
// The kernel is built from the step functions of abr_step.cu (head, advance_trace, position_of, lookup_tables,
// reset_seg_phase, the policy rules, session_knobs and env_knobs), not a restatement of them: this unit compiles that
// file's device part (ABR_STEP_DEVICE_ONLY).  A unit of its own, so that the module of the step kernels stays as it was.
#define ABR_STEP_DEVICE_ONLY
#include "abr_step.cu"

namespace abr {

namespace {

constexpr int kSharedWarps = 4;                    // links per block
constexpr int kSharedSmemMax = 200 * 1024;         // dynamic shared memory the staged path may use per block
enum : int { kWaiting = 0, kActive = 1, kFinished = 2 };

__device__ __forceinline__ double warp_min(double x) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x = fmin(x, __shfl_xor_sync(0xffffffffu, x, o));
    return x;
}

// Bytes of one warp's staged rows: C (with the slack the head reads past C[T]) and the bucket index.
__host__ __device__ __forceinline__ size_t shared_cum_bytes(int T_max) {
    return ((size_t)cum_smem_doubles(T_max) * 8u + 15u) & ~(size_t)15u;
}
__host__ __device__ __forceinline__ size_t shared_slice_bytes(int T_max) {
    return shared_cum_bytes(T_max) + (size_t)idx_stride(T_max) * 2u;
}

// SPEC §4 action of a player's download k from its own state and knobs kn (SPEC §4.7).  DYNAMIC updates `mode`.
template <bool SMEM>
__device__ __forceinline__ int shared_action(const EnvView& v, const SharedRun& r, const Sess& s, const int pol,
                                             const SessKnobs& kn, const int i, const int k, uint32_t& mode,
                                             bool& flagged) {
    const int A = v.A;
    if (pol == ABR_POLICY_FIXED) {
        int a = __ldg(r.actions_in + (size_t)k * (size_t)v.n + i);
        if (a < 0 || a >= A) { flagged = true; a = a < 0 ? 0 : A - 1; }
        return a;
    }
    if (pol == ABR_POLICY_RANDOM) {   // counter (session, k / 8), 16-bit slice k % 8 (low half of word 0 first)
        const unsigned long long g = (unsigned long long)(v.session_base + i);
        const uint4 x = philox4x32_10((uint32_t)g, (uint32_t)(g >> 32), (uint32_t)k >> 3, 0u, r.seed_lo, r.seed_hi);
        const uint32_t m = (uint32_t)k & 7u;
        const uint32_t w = (m >> 1) == 0 ? x.x : (m >> 1) == 1 ? x.y : (m >> 1) == 2 ? x.z : x.w;
        return (int)((((w >> (16u * (m & 1u))) & 0xffffu) * (uint32_t)A) >> 16);
    }
    if (pol == ABR_POLICY_BBA) return policy_bba(v, kn, s.buffer);
    if (s.done) return 0;   // chunk == V: no sizes row (the download is inert; DYNAMIC keeps its rule)
    const int row = s.chunk * A;
    ABR_CHECK(s.chunk >= 0 && s.chunk < v.V, "policy row");
    auto size_at = [&](const int a) -> double {
        return SMEM ? lds_f64(s.tab_s + 16u * (uint32_t)(row + a)) : __ldg(&s.tab[row + a].x);
    };
    if (pol == ABR_POLICY_DYNAMIC) {
        mode = (uint32_t)dynamic_mode(kn, s.chunk, s.buffer, (int)mode);
        if (mode) return policy_bola(v, kn, s.buffer, row, size_at);
        return policy_rate(v, kn, i, s.hist_len, size_at);
    }
    if (pol == ABR_POLICY_RATE) return policy_rate(v, kn, i, s.hist_len, size_at);
    return policy_bola(v, kn, s.buffer, row, size_at);
}

template <bool SMEM>
__global__ void __launch_bounds__(32 * kSharedWarps, 1)
abr_shared_kernel(EnvView v, SharedRun r) {
    extern __shared__ __align__(16) double2 s_tab2[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int link = blockIdx.x * kSharedWarps + warp;
    const int G = r.G;
    const bool live_link = link < r.n_links;                  // warp-uniform
    const int i0 = live_link ? link * G : 0;
    const bool valid = live_link && lane < G;                 // a player; the other lanes follow the link only
    const int i = valid ? i0 + lane : i0;
    // SPEC §2 for the link: its trace and start position (every player of the link counts a bad trace id or offset)
    int n_bad = 0;
    int tr = live_link ? __ldg(r.link_trace_id + link) : 0;
    if (tr < 0 || tr >= v.n_traces) { ++n_bad; tr = 0; }
    const double off = (live_link && r.link_offset) ? __ldg(r.link_offset + link) : 0.0;
    RawState w;
    w.tr = tr; w.seg = 0; w.chunk = 0; w.last_q = v.p.default_quality; w.phi = 0.0; w.pos = 0.0; w.buffer = 0.0;
    Sess s;
    make_sess(v, i, w, s);
    reset_seg_phase(s.I, s.T, off, s.seg, s.phi, n_bad);
    s.done = false; s.hist_len = 0;
    if (SMEM) {
        double2* s_tab = s_tab2;
        const int tab_n = v.V * v.A;
        for (int j = threadIdx.x; j < tab_n; j += blockDim.x) s_tab[j] = __ldg(v.tab + j);
        char* slice = reinterpret_cast<char*>(s_tab + tab_n) + (size_t)warp * shared_slice_bytes(v.T_max);
        double* s_cum = reinterpret_cast<double*>(slice);
        uint32_t* s_idx = reinterpret_cast<uint32_t*>(slice + shared_cum_bytes(v.T_max));
        const int cs = cum_stride(v.T_max), is = idx_stride(v.T_max) / 2;
        const double* g_cum = v.trace_cum + (size_t)tr * cs;
        const uint32_t* g_idx = reinterpret_cast<const uint32_t*>(v.trace_idx + (size_t)tr * idx_stride(v.T_max));
        for (int j = lane; j < cs; j += 32) s_cum[j] = __ldg(g_cum + j);
        if (lane < cum_smem_doubles(v.T_max) - cs) s_cum[cs + lane] = __longlong_as_double(0x7ff0000000000000ll);
        for (int j = lane; j < is; j += 32) s_idx[j] = __ldg(g_idx + j);
        __syncthreads();
        s.cum_s = (uint32_t)__cvta_generic_to_shared(s_cum);
        s.idx_s = (uint32_t)__cvta_generic_to_shared(s_idx);
        s.tab_s = (uint32_t)__cvta_generic_to_shared(s_tab);
#ifdef ABR_CHECKED
        s.chk_cum_n = cum_smem_doubles(v.T_max); s.chk_idx_n = idx_stride(v.T_max);
#endif
    }
    if (!live_link) return;                                   // after the block's only barrier
    s.pos = position_of<SMEM>(s, s.seg, s.phi);
    const double pos_start = s.pos;

    const AbrParams& p = v.p;
    const int steps = r.steps, V = v.V, A = v.A;
    const size_t N = (size_t)v.n, cap = (size_t)v.cap;
    const bool hist = p.track_history != 0, prev_ladder = p.smooth_prev_ladder != 0;
    const double inv_q = pow2_inverse(p.sleep_quantum);
    const uint32_t pw = (lane >> 3) == 0 ? r.policy[0] : (lane >> 3) == 1 ? r.policy[1] : (lane >> 3) == 2 ? r.policy[2] : r.policy[3];
    const int pol = valid ? (int)((pw >> (4 * (lane & 7))) & 0xfu) : ABR_POLICY_FIXED;
    // the player's knobs: its own while per-session knobs are installed, the environment-wide ones otherwise
    SessKnobs kn = env_knobs(v);
    if (valid && v.sp.on) {
        if (pol == ABR_POLICY_BBA) kn = session_knobs<ABR_POLICY_BBA>(v, i);
        else if (pol == ABR_POLICY_RATE) kn = session_knobs<ABR_POLICY_RATE>(v, i);
        else if (pol == ABR_POLICY_BOLA) kn = session_knobs<ABR_POLICY_BOLA>(v, i);
        else if (pol == ABR_POLICY_DYNAMIC) kn = session_knobs<ABR_POLICY_DYNAMIC>(v, i);
    }
    uint32_t mode = (valid && pol == ABR_POLICY_DYNAMIC) ? v.pol.dyn_mode[i] : 0u;
    bool flagged = false;
    // the player: its state in the event loop, its download in flight and the request snapshot of the link
    int state = kWaiting, k = 0, q = 0, seg_req = 0;
    double wait = 0.0, rem = 0.0, phi_req = 0.0, periods_req = 0.0, req_time = 0.0;
    Lookup lk{};
    if (valid) {
        wait = r.join_delay ? __ldg(r.join_delay + i) : 0.0;
        if (!(wait >= 0.0 && wait <= 1.7976931348623157e308)) { flagged = true; wait = 0.0; }   // negative, NaN, inf
    }
    if (!valid || steps == 0) state = kFinished;
    double rew = 0.0, reb = 0.0, su = 0.0, sm = 0.0, sl = 0.0, dl = 0.0;
    int n_steps = 0, n_eps = 0;
    double clock = 0.0, periods = 0.0, delivered = 0.0;
    const StepOutputs<double>& o = r.traj;

    auto requests = [&]() {
        while (state == kWaiting && wait <= 0.0) {
            if (k >= steps) { state = kFinished; break; }   // the sleep after the last download is over
            q = shared_action<SMEM>(v, r, s, pol, kn, i, k, mode, flagged);
            req_time = clock;
            if (!p.auto_reset && s.done) {   // SPEC §3's inert step: no link time, counts as a download
                const size_t ix = (size_t)k * N + i;
                if (o.delay) o.delay[ix] = 0.0;
                if (o.sleep) o.sleep[ix] = 0.0;
                if (o.buffer) o.buffer[ix] = s.buffer;
                if (o.rebuf) o.rebuf[ix] = 0.0;
                if (o.reward) o.reward[ix] = 0.0;
                if (o.eov) o.eov[ix] = 1;
                if (o.actions) o.actions[ix] = q;
                if (r.request_time) r.request_time[ix] = req_time;
                if (++k >= steps) state = kFinished;
                continue;
            }
            lk = lookup_tables<SMEM>(s, A, V, s.chunk, q, s.last_q, prev_ladder);
            rem = lk.size;
            seg_req = s.seg; phi_req = s.phi; periods_req = periods;
            state = kActive;
        }
    };

    requests();
    const long long max_events = (long long)G * (2ll * steps + 1) + 1;   // every event brings a rem or a wait to 0 (SPEC §9)
    long long events = 0;
    for (;;) {
        const unsigned act = __ballot_sync(0xffffffffu, state == kActive);
        const unsigned wt = __ballot_sync(0xffffffffu, state == kWaiting);
        if ((act | wt) == 0u) break;
        if (++events > max_events) { if (state != kFinished) flagged = true; break; }   // safety net, never expected
        const int n = __popc(act);
        const double inf = __longlong_as_double(0x7ff0000000000000ll);
        const double m = warp_min(state == kActive ? rem : inf);
        const double tw = warp_min(state == kWaiting ? wait : inf);
        Head h{};
        double phi_new = 0.0, dc = inf;
        if (n > 0) {   // where the smallest download would complete: n*m more data at an equal share
            bool werr = false;
            head<SMEM>(s, dadd(s.pos, dmul((double)n, m)), h, werr);
            phi_new = ddiv(dsub(h.target, h.c_j), dsub(h.c_j1, h.c_j));
            dc = max0d(dmul(dadd(dadd(diff2double(h.j, s.seg), h.kx), dsub(phi_new, s.phi)), s.I));
            if (werr && state == kActive) flagged = true;
        }
        double dt;
        if (n > 0 && dc <= tw) {   // completion event
            dt = dc;
            s.seg = h.j; s.phi = phi_new; s.pos = h.target;
            periods = dadd(periods, ddiv(h.kx, s.Td));   // exact: kx = whole periods * T
            if (state == kActive) rem = dsub(rem, m);
        } else {                   // arrival event: the link moves as SPEC §3.3 moves it for a sleep
            dt = tw;
            const int seg0 = s.seg;
            const double pos0 = s.pos;
            const double nx = floor(dadd(s.phi, s.inv_I != 0.0 ? dmul(tw, s.inv_I) : ddiv(tw, s.I)));   // advance_trace's n
            advance_trace(s.seg, s.phi, tw, s.I, s.inv_I, s.T);
            s.pos = position_of<SMEM>(s, s.seg, s.phi);
            double crossed;   // (seg0 + nx) div T: whole trace periods the advance crossed
            if (nx < 2147480000.0) {
                crossed = (double)(((unsigned)seg0 + (unsigned)(int)nx) / (unsigned)s.T);
            } else {          // exact while nx < 2^53: nx - r is a multiple of T
                const double r0 = fmod(nx, s.Td);
                crossed = dadd(ddiv(dsub(nx, r0), s.Td), dadd((double)seg0, r0) >= s.Td ? 1.0 : 0.0);
            }
            periods = dadd(periods, crossed);
            if (n > 0 && state == kActive) rem = dsub(rem, ddiv(dadd(dsub(s.pos, pos0), dmul(crossed, s.P)), (double)n));
        }
        if (state == kWaiting) wait = dsub(wait, dt);
        clock = dadd(clock, dt);
        // completions, SPEC §3.1 (delay) and §3.2-§3.5, except that the sleep is a wait of the player's own
        const bool done_now = state == kActive && rem <= 0.0;
        if (done_now) {
            const double kd = dadd(diff2double(s.seg, seg_req), dmul(dsub(periods, periods_req), s.Td));
            const double delay = dadd(max0d(dmul(dadd(kd, dsub(s.phi, phi_req)), s.I)), p.rtt);
            const double thr = hist ? ddiv(lk.size, delay) : 0.0;
            double rebuf, buffer, sleep = 0.0;
            {   // max(delay - buffer, 0) and max(buffer - delay, 0) + L, as step_tail forms them
                const double d = dsub(delay, s.buffer);
                const int hi = __double2hiint(d), lo = __double2loint(d);
                const int neg = hi >> 31;
                rebuf = __hiloint2double(hi & ~neg, lo & ~neg);
                buffer = dadd(__hiloint2double((hi ^ (int)0x80000000u) & neg, lo & neg), p.chunk_length);
            }
            if (buffer > p.max_buffer) {
                const double over = dsub(buffer, p.max_buffer);
                sleep = dmul(ceil(inv_q != 0.0 ? dmul(over, inv_q) : ddiv(over, p.sleep_quantum)), p.sleep_quantum);
                buffer = dsub(buffer, sleep);
            }
            const double smooth = fabs(dsub(lk.u, lk.u_prev));
            const double reward = dsub(dsub(lk.u, dmul(p.rebuf_penalty, rebuf)), dmul(p.smooth_penalty, smooth));
            s.hist_len += 1;
            s.last_q = q;
            s.chunk += 1;
            s.buffer = buffer;
            const bool eov = s.chunk >= V;
            bool wrapped = false;
            if (eov) {
                if (p.auto_reset) { s.chunk = 0; s.buffer = 0.0; s.last_q = p.default_quality; s.hist_len = 0; wrapped = true; }
                else s.done = true;
            }
            rew = dadd(rew, reward); reb = dadd(reb, rebuf); su = dadd(su, lk.u);
            sm = dadd(sm, smooth); sl = dadd(sl, sleep); dl = dadd(dl, delay);
            n_steps += 1; n_eps += eov ? 1 : 0;
            if (!wrapped && hist) v.bw_hist[(size_t)((s.hist_len - 1) % v.K) * cap + i] = thr;
            const size_t ix = (size_t)k * N + i;
            if (o.delay) o.delay[ix] = delay;
            if (o.sleep) o.sleep[ix] = sleep;
            if (o.buffer) o.buffer[ix] = buffer;
            if (o.rebuf) o.rebuf[ix] = rebuf;
            if (o.reward) o.reward[ix] = reward;
            if (o.eov) o.eov[ix] = eov ? 1 : 0;
            if (o.actions) o.actions[ix] = q;
            if (r.request_time) r.request_time[ix] = req_time;
            wait = sleep;   // the player leaves the link once it has waited out the sleep after its last download
            state = kWaiting;
            ++k;
        }
        // the data delivered, summed in completion order (players in lane order within an event)
        for (unsigned cm = __ballot_sync(0xffffffffu, done_now); cm; cm &= cm - 1u)
            delivered = dadd(delivered, __shfl_sync(0xffffffffu, lk.size, __ffs(cm) - 1));
        requests();
    }
    if (lane == 0) {
        if (r.link_time) r.link_time[link] = clock;
        if (r.link_capacity) r.link_capacity[link] = dsub(dadd(dmul(periods, s.P), s.pos), pos_start);
        if (r.link_delivered) r.link_delivered[link] = delivered;
    }
    if (!valid) return;
    const int n_err = n_bad + (flagged ? 1 : 0);
    if (n_err) atomicAdd(v.errors, (unsigned long long)n_err);
    // the state of a fresh run (what abr_env_run leaves), with the link's final position
    v.trace_id[i] = tr; v.seg[i] = s.seg; v.phi[i] = s.phi; v.pos[i] = s.pos;
    v.chunk[i] = s.chunk; v.last_q[i] = s.last_q; v.buffer[i] = s.buffer; v.done[i] = s.done ? 1 : 0;
    v.hist_len[i] = hist ? s.hist_len : 0;
    v.last_pred[i] = 0.0; v.err_len[i] = 0;
    v.t_now[i] = 0.0; v.play_time[i] = 0.0; v.started[i] = p.start_up_length <= 0.0 ? 1 : 0;
    v.play_id[i] = 0; v.play_len[i] = 0.0;
    if (pol == ABR_POLICY_DYNAMIC) v.pol.dyn_mode[i] = (uint8_t)mode;
    const double add[ABR_NUM_ACC] = {rew, reb, su, sm, sl, dl, (double)n_steps, (double)n_eps, 0.0, 0.0, 0.0};
#pragma unroll
    for (int j = 0; j < ABR_NUM_ACC; ++j) v.acc[(size_t)j * cap + i] = dadd(0.0, add[j]);
    // Simulator.calculate_qoe outside live mode (session_cost of the episode kernel)
    if (r.qoe_cost) r.qoe_cost[i] = dadd(dmul(p.rebuf_penalty, dadd(0.0, reb)), dmul(p.smooth_penalty, dadd(0.0, sm)));
}

// Dynamic shared memory of the staged path, or 0 for the global path: traces without a bucket index (longer than
// 65 535 segments) and rows that do not fit.
size_t shared_smem_bytes(const EnvView& v) {
    if (v.T_max > kIdxMaxT) return 0;
    const size_t b = (size_t)v.V * (size_t)v.A * 16u + (size_t)kSharedWarps * shared_slice_bytes(v.T_max);
    return b <= (size_t)kSharedSmemMax ? b : 0;
}

}  // namespace

cudaError_t launch_shared(const EnvView& v, const SharedRun& r, cudaStream_t st) {
    if (r.n_links == 0) return cudaSuccess;
    const int blocks = (r.n_links + kSharedWarps - 1) / kSharedWarps;
    const size_t smem = shared_smem_bytes(v);
    if (smem) {
        cudaError_t e = cudaFuncSetAttribute(abr_shared_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        abr_shared_kernel<true><<<blocks, 32 * kSharedWarps, smem, st>>>(v, r);
    } else {
        abr_shared_kernel<false><<<blocks, 32 * kSharedWarps, 0, st>>>(v, r);
    }
    count_launch();
    return cudaGetLastError();
}

}  // namespace abr
