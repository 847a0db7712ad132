// C-ABI of libabr_b200.so (declared in include/abr_b200.h): handle management, validation,
// host<->device plumbing.  No compute happens on the CPU here: every entry point either launches
// the sm_100a kernels of abr_step.cu / abr_mpc.cu or fails with ABR_ERR_CUDA.
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <new>
#include <vector>

#include "abr_common.cuh"
#include "../../include/abr_b200_lookahead.h"
#include "../../include/abr_b200_mpc_pred.h"
#include "../../include/abr_b200_mpc_scen.h"
#include "../../include/abr_b200_obs.h"

namespace abr {
static std::atomic<long long> g_launches{0};
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
}  // namespace abr

using namespace abr;

static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CUDA_TRY(expr)                                                                                 \
    do {                                                                                               \
        cudaError_t _e = (expr);                                                                       \
        if (_e != cudaSuccess) return fail(ABR_ERR_CUDA, "%s: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                                           __FILE__, __LINE__);                                        \
    } while (0)

// Grow-only device memory on the current device.  Growing (or moving to another device) first waits for the device,
// since work already launched may still use the old block; it then allocates half again what was asked for.
struct DeviceBuffer {
    void* p = nullptr;
    size_t bytes = 0;
    int device = -1;
    DeviceBuffer() = default;
    DeviceBuffer(const DeviceBuffer&) = delete;
    DeviceBuffer& operator=(const DeviceBuffer&) = delete;
    ~DeviceBuffer() { if (p) cudaFree(p); }
    // at least `want` bytes; *fresh (nullable) tells whether this call allocated a new block
    cudaError_t reserve(size_t want, bool* fresh = nullptr) {
        if (fresh) *fresh = false;
        int dev = 0;
        cudaError_t e = cudaGetDevice(&dev);
        if (e != cudaSuccess || (p && dev == device && want <= bytes)) return e;
        if (p) { cudaDeviceSynchronize(); cudaFree(p); p = nullptr; bytes = 0; }
        const size_t n = want + want / 2 > 256 ? want + want / 2 : 256;
        e = cudaMalloc(&p, n);
        if (e != cudaSuccess) { p = nullptr; return e; }
        bytes = n; device = dev;
        if (fresh) *fresh = true;
        return cudaSuccess;
    }
    template <typename T>
    T* as() const { return static_cast<T*>(p); }
};

struct AbrEnv {
    EnvView v{};
    int device = 0;
    std::vector<void*> allocs;
    double* d_stats_partials = nullptr;
    int n_partials_cap = 0;
    bool was_reset = false;   // abr_env_reset has run (an empty batch, n == 0, is legal and makes every call a no-op)
    uint32_t step_base = 0;   // fused-episode steps since the last reset: offsets the random policy's counter (SPEC §4)
    int32_t* d_perm = nullptr;   // session order installed by abr_env_set_order (capacity entries), v.perm points here when set
    int n_order = 0;
    DeviceBuffer sort_hist;   // (trace, run) cells of abr_env_reset_sorted's counting sort, zero between calls
    DeviceBuffer sort_scan;   // the scan's scratch of that sort
    int fresh_partials = 0;   // > 0: d_stats_partials holds that many block sums of the current accumulators
    double* d_stats_out = nullptr;
    uint32_t* d_draw_counter = nullptr;       // draws of abr_env_step_policy since the last reset
    StatsScratch stats_scratch;               // group sums and the counters of finished blocks / groups (zero between launches)
    // scratch for the *_host entry points
    int32_t* d_trace_id = nullptr;
    double* d_offset = nullptr;
    DeviceBuffer actions, reward_traj;        // abr_env_run_host's [steps][N] actions in and reward trajectory out
    double bola_vmax = 0.0;   // max over the log table of SPEC §4.3 (when every size is > 0, i.e. v.pol.bola_v is set)

    ~AbrEnv() {
        for (void* p : allocs) cudaFree(p);
    }
    template <typename T>
    cudaError_t alloc(T** out, size_t count) {
        void* p = nullptr;
        cudaError_t e = cudaMalloc(&p, (count ? count : 1) * sizeof(T));
        if (e == cudaSuccess) { allocs.push_back(p); *out = (T*)p; }
        return e;
    }
};

// The calls that take host tables validate them first, so that bad arguments are reported without a device.
static int require_device() {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(ABR_ERR_CUDA, "no CUDA device: this library has no CPU fallback");
    }
    return ABR_OK;
}

extern "C" {

int abr_version(void) { return ABR_VERSION; }
const char* abr_last_error(void) { return g_err; }
long long abr_launch_count(void) { return g_launches.load(); }

int abr_device_info(int* sm_count, int* cc_major, int* cc_minor, long long* total_mem_bytes) {
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, dev));
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (cc_major) *cc_major = prop.major;
    if (cc_minor) *cc_minor = prop.minor;
    if (total_mem_bytes) *total_mem_bytes = (long long)prop.totalGlobalMem;
    return ABR_OK;
}

void abr_params_default(AbrParams* p) {
    if (!p) return;
    memset(p, 0, sizeof(*p));
    p->chunk_length = 4.0; p->max_buffer = 60.0; p->rtt = 0.08; p->payload = 0.95; p->sleep_quantum = 0.5;
    p->rebuf_penalty = 4.3; p->smooth_penalty = 1.0; p->utility_scale = 0.001;
    p->bba_reservoir = 5.0; p->bba_cushion = 10.0;
    p->start_up_length = 0.0; p->startup_penalty = 0.0; p->latency_penalty = 0.0; p->latency_tick = 0.01;
    p->utility_mode = 0; p->default_quality = 1; p->auto_reset = 1; p->hist_k = 5;
    p->track_history = 0; p->track_acc = 0; p->live = 0; p->smooth_prev_ladder = 0;
}

static int check_params(const AbrParams* p, int A) {
    if (!p) return fail(ABR_ERR_INVALID, "params is NULL");
    if (!(p->chunk_length > 0.0) || !std::isfinite(p->chunk_length)) return fail(ABR_ERR_INVALID, "chunk_length must be > 0");
    if (!(p->max_buffer > 0.0)) return fail(ABR_ERR_INVALID, "max_buffer must be > 0");
    if (!(p->payload > 0.0) || !std::isfinite(p->payload)) return fail(ABR_ERR_INVALID, "payload must be > 0");
    if (!(p->rtt >= 0.0) || !std::isfinite(p->rtt)) return fail(ABR_ERR_INVALID, "rtt must be >= 0");
    if (!(p->sleep_quantum > 0.0)) return fail(ABR_ERR_INVALID, "sleep_quantum must be > 0");
    if (p->hist_k < 1 || p->hist_k > 64) return fail(ABR_ERR_RANGE, "hist_k must be in [1, 64]");
    if (p->default_quality >= A) return fail(ABR_ERR_RANGE, "default_quality %d out of range for A=%d", p->default_quality, A);
    if (p->utility_mode != 0 && p->utility_mode != 1) return fail(ABR_ERR_INVALID, "utility_mode must be 0 or 1");
    if (!(p->bba_cushion > 0.0)) return fail(ABR_ERR_INVALID, "bba_cushion must be > 0");
    if (p->live && !(p->start_up_length <= p->max_buffer))
        return fail(ABR_ERR_INVALID, "live mode needs start_up_length <= max_buffer (the start-up phase could never end)");
    if (!std::isfinite(p->start_up_length) || !std::isfinite(p->startup_penalty) || !std::isfinite(p->latency_penalty))
        return fail(ABR_ERR_INVALID, "start_up_length / startup_penalty / latency_penalty must be finite");
    if (!(p->latency_tick > 0.0) || !std::isfinite(p->latency_tick)) return fail(ABR_ERR_INVALID, "latency_tick must be finite and > 0");
    return ABR_OK;
}

static void utility_table(const double* bitrates, int V, int A, const AbrParams* p, std::vector<double>& util) {
    util.resize((size_t)V * A);
    for (int v = 0; v < V; ++v)
        for (int a = 0; a < A; ++a) {
            const double b = bitrates[(size_t)v * A + a];
            util[(size_t)v * A + a] = p->utility_mode == 1 ? std::log(b / bitrates[(size_t)v * A + A - 1])  // mpc.py:99-102
                                                           : b * p->utility_scale;                        // mpc.py:95-97
        }
}

void abr_policy_params_default(AbrPolicyParams* p) {
    if (!p) return;
    p->rb_safety = 1.0; p->bola_min_buffer = 10.0; p->bola_target_buffer = 30.0;
}

static int check_policy_params(const AbrPolicyParams* pp) {
    if (!pp) return fail(ABR_ERR_INVALID, "policy params is NULL");
    if (!(pp->rb_safety > 0.0) || !std::isfinite(pp->rb_safety)) return fail(ABR_ERR_INVALID, "rb_safety must be finite and > 0");
    if (!(pp->bola_min_buffer > 0.0) || !std::isfinite(pp->bola_min_buffer) || !std::isfinite(pp->bola_target_buffer) ||
        !(pp->bola_min_buffer < pp->bola_target_buffer))
        return fail(ABR_ERR_INVALID, "need 0 < bola_min_buffer < bola_target_buffer, both finite");
    return ABR_OK;
}

// SPEC §4.2 / §4.3 parameters (already validated): BOLA's (Vp, gp) derived from the buffer range as dash.js does
static void install_policy_params(AbrEnv* env, const AbrPolicyParams* pp) {
    EnvView::Policy& pol = env->v.pol;
    pol.rb_safety = pp->rb_safety;
    pol.bola_vmax = env->bola_vmax;
    pol.bola_gp = env->bola_vmax / (pp->bola_target_buffer / pp->bola_min_buffer - 1.0);
    pol.bola_Vp = pp->bola_min_buffer / pol.bola_gp;
}

static int check_tables(const double* sizes, const double* bitrates, int V, int A) {
    if (!sizes || !bitrates) return fail(ABR_ERR_INVALID, "sizes/bitrates is NULL");
    if (V < 1 || A < 1 || A > 16) return fail(ABR_ERR_RANGE, "need V >= 1 and 1 <= A <= 16 (got V=%d A=%d)", V, A);
    for (size_t i = 0; i < (size_t)V * A; ++i) {
        if (!std::isfinite(sizes[i]) || sizes[i] < 0.0) return fail(ABR_ERR_INVALID, "sizes[%zu] = %g is not finite and >= 0", i, sizes[i]);
        if (!std::isfinite(bitrates[i])) return fail(ABR_ERR_INVALID, "bitrates[%zu] is not finite", i);
    }
    return ABR_OK;
}

int abr_env_create(const double* h_trace_bw, const int32_t* h_trace_len, const double* h_trace_interval, int n_traces,
                   int T_max, const double* h_sizes, const double* h_bitrates, int V, int A, const AbrParams* params,
                   int max_sessions, AbrEnv** out) {
    if (!out) return fail(ABR_ERR_INVALID, "out is NULL");
    *out = nullptr;
    if (!h_trace_bw || !h_trace_len || !h_trace_interval) return fail(ABR_ERR_INVALID, "trace table is NULL");
    if (n_traces < 1 || T_max < 1 || max_sessions < 1) return fail(ABR_ERR_RANGE, "n_traces, T_max, max_sessions must be >= 1");
    int rc = check_tables(h_sizes, h_bitrates, V, A);
    if (rc) return rc;
    rc = check_params(params, A);
    if (rc) return rc;
    for (int t = 0; t < n_traces; ++t) {
        const int len = h_trace_len[t];
        if (len < 1 || len > T_max) return fail(ABR_ERR_RANGE, "trace_len[%d] = %d not in [1, %d]", t, len, T_max);
        if (!(h_trace_interval[t] > 0.0) || !std::isfinite(h_trace_interval[t]))
            return fail(ABR_ERR_INVALID, "trace_interval[%d] must be finite and > 0", t);
        for (int i = 0; i < len; ++i) {
            const double b = h_trace_bw[(size_t)t * T_max + i];
            if (!(b > 0.0) || !std::isfinite(b))  // the reference would divide by zero / never finish (D14)
                return fail(ABR_ERR_INVALID, "trace %d segment %d: bandwidth %g must be finite and > 0", t, i, b);
        }
    }
    if (int rc = require_device()) return rc;
    AbrEnv* e = new (std::nothrow) AbrEnv();
    if (!e) return fail(ABR_ERR_INVALID, "out of host memory");
    struct Guard { AbrEnv* e; ~Guard() { delete e; } } guard{e};
    CUDA_TRY(cudaGetDevice(&e->device));
    EnvView& v = e->v;
    v.n_traces = n_traces; v.T_max = T_max; v.V = V; v.A = A; v.K = params->hist_k; v.cap = max_sessions; v.n = 0;
    v.session_base = 0; v.p = *params;
    const size_t cap = (size_t)max_sessions;
    double *d_bw, *d_int, *d_sizes, *d_util;
    int32_t* d_len;
    CUDA_TRY(e->alloc(&d_bw, (size_t)n_traces * T_max));
    CUDA_TRY(e->alloc(&d_len, n_traces));
    CUDA_TRY(e->alloc(&d_int, n_traces));
    CUDA_TRY(e->alloc(&d_sizes, (size_t)V * A));
    CUDA_TRY(e->alloc(&d_util, (size_t)V * A));
    std::vector<double> util;
    utility_table(h_bitrates, V, A, params, util);
    CUDA_TRY(cudaMemcpy(d_bw, h_trace_bw, sizeof(double) * n_traces * T_max, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(d_len, h_trace_len, sizeof(int32_t) * n_traces, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(d_int, h_trace_interval, sizeof(double) * n_traces, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(d_sizes, h_sizes, sizeof(double) * V * A, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(d_util, util.data(), sizeof(double) * V * A, cudaMemcpyHostToDevice));
    v.trace_bw = d_bw; v.trace_len = d_len; v.trace_interval = d_int; v.sizes = d_sizes; v.util = d_util;
    v.uniform_util = 1;   // bitwise: the kernels may then carry a step's utility over as the next step's "previous" one
    for (size_t i = (size_t)A; i < (size_t)V * A; ++i)
        if (memcmp(&util[i], &util[i % A], sizeof(double)) != 0) { v.uniform_util = 0; break; }
    {   // packed {size, utility} table for the step kernels
        std::vector<double> tab(2 * (size_t)V * A);
        for (size_t i = 0; i < (size_t)V * A; ++i) { tab[2 * i] = h_sizes[i]; tab[2 * i + 1] = util[i]; }
        double* d_tab;
        CUDA_TRY(e->alloc(&d_tab, tab.size()));
        CUDA_TRY(cudaMemcpy(d_tab, tab.data(), sizeof(double) * tab.size(), cudaMemcpyHostToDevice));
        v.tab = reinterpret_cast<const double2*>(d_tab);
    }
    {   // BOLA's utilities v[k][a] = log(sizes[k][a] / sizes[k][0]) (SPEC §4.3), with the C library's log like the
        // utility table; only when every size is > 0 (else BOLA calls fail and the table is not needed)
        bool positive = true;
        for (size_t i = 0; i < (size_t)V * A && positive; ++i) positive = h_sizes[i] > 0.0;
        if (positive) {
            std::vector<double> lv((size_t)V * A);
            double vmax = -INFINITY;
            for (int k = 0; k < V; ++k)
                for (int a = 0; a < A; ++a) {
                    const double x = std::log(h_sizes[(size_t)k * A + a] / h_sizes[(size_t)k * A]);
                    lv[(size_t)k * A + a] = x;
                    if (x > vmax) vmax = x;
                }
            double* d_v;
            CUDA_TRY(e->alloc(&d_v, lv.size()));
            CUDA_TRY(cudaMemcpy(d_v, lv.data(), sizeof(double) * lv.size(), cudaMemcpyHostToDevice));
            v.pol.bola_v = d_v;
            e->bola_vmax = vmax;
        }
        AbrPolicyParams pp;
        abr_policy_params_default(&pp);
        install_policy_params(e, &pp);
    }
    // per-trace tables of SPEC §3.1 (cumulative capacity, search widths), built on the device
    // (+4 doubles of slack: the step reads C[j .. j+4] and discards what lies past its candidates)
    double* d_cum;
    int32_t* d_ok;
    CUDA_TRY(e->alloc(&d_cum, (size_t)n_traces * cum_stride(T_max) + 4));
    CUDA_TRY(cudaMemset(d_cum + (size_t)n_traces * cum_stride(T_max), 0, 4 * sizeof(double)));
    CUDA_TRY(e->alloc(&d_ok, n_traces));
    TraceMeta* d_meta;
    CUDA_TRY(e->alloc(&d_meta, n_traces));
    uint16_t* d_idx;
    CUDA_TRY(e->alloc(&d_idx, (size_t)n_traces * idx_stride(T_max) + 8));
    v.trace_cum = d_cum; v.trace_meta = d_meta; v.trace_idx = d_idx;
    CUDA_TRY(launch_trace_table(v, d_cum, d_idx, d_ok, d_meta, 0));
    {
        std::vector<int32_t> bits(n_traces);
        CUDA_TRY(cudaMemcpy(bits.data(), d_ok, sizeof(int32_t) * n_traces, cudaMemcpyDeviceToHost));
        for (int t = 0; t < n_traces; ++t)
            if (bits[t] <= 0)
                return fail(ABR_ERR_INVALID, "trace %d: every segment capacity bandwidth*payload*interval must be representable "
                                             "next to the capacity of the whole trace period (positive, finite)", t);
    }
    CUDA_TRY(e->alloc(&v.seg, cap)); CUDA_TRY(e->alloc(&v.chunk, cap)); CUDA_TRY(e->alloc(&v.last_q, cap));
    CUDA_TRY(e->alloc(&v.trace_id, cap)); CUDA_TRY(e->alloc(&v.hist_len, cap)); CUDA_TRY(e->alloc(&v.err_len, cap));
    CUDA_TRY(e->alloc(&v.done, cap)); CUDA_TRY(e->alloc(&v.phi, cap)); CUDA_TRY(e->alloc(&v.buffer, cap));
    CUDA_TRY(e->alloc(&v.pos, cap));
    CUDA_TRY(e->alloc(&v.started, cap)); CUDA_TRY(e->alloc(&v.t_now, cap)); CUDA_TRY(e->alloc(&v.play_time, cap));
    CUDA_TRY(e->alloc(&v.play_id, cap)); CUDA_TRY(e->alloc(&v.play_len, cap));
    CUDA_TRY(e->alloc(&v.bw_hist, cap * v.K)); CUDA_TRY(e->alloc(&v.last_pred, cap));
    CUDA_TRY(e->alloc(&v.err_ring, cap * v.K)); CUDA_TRY(e->alloc(&v.acc, cap * ABR_NUM_ACC));
    CUDA_TRY(e->alloc(&v.errors, 1));
    CUDA_TRY(cudaMemset(v.errors, 0, sizeof(unsigned long long)));
    CUDA_TRY(cudaMemset(v.bw_hist, 0, sizeof(double) * cap * v.K));
    CUDA_TRY(cudaMemset(v.err_ring, 0, sizeof(double) * cap * v.K));
    e->n_partials_cap = stats_num_partials(max_sessions) > rollout_num_blocks(max_sessions)
                            ? stats_num_partials(max_sessions) : rollout_num_blocks(max_sessions);
    CUDA_TRY(e->alloc(&e->d_stats_partials, (size_t)e->n_partials_cap * ABR_NUM_ACC));
    CUDA_TRY(e->alloc(&e->d_stats_out, ABR_NUM_STATS));
    CUDA_TRY(e->alloc(&e->d_draw_counter, 1));
    CUDA_TRY(cudaMemset(e->d_draw_counter, 0, sizeof(uint32_t)));
    {
        const int n_groups = stats_num_groups(e->n_partials_cap);
        CUDA_TRY(e->alloc(&e->stats_scratch.group_partials, (size_t)n_groups * ABR_NUM_ACC));
        CUDA_TRY(e->alloc(&e->stats_scratch.counters, (size_t)n_groups + 1));
        CUDA_TRY(cudaMemset(e->stats_scratch.counters, 0, sizeof(unsigned int) * ((size_t)n_groups + 1)));
    }
    CUDA_TRY(e->alloc(&e->d_trace_id, cap));
    CUDA_TRY(e->alloc(&e->d_offset, cap));
    guard.e = nullptr;
    *out = e;
    return ABR_OK;
}

void abr_env_destroy(AbrEnv* env) { delete env; }

int abr_env_num_sessions(const AbrEnv* env) { return env ? env->v.n : 0; }

int abr_sort_by_trace(const int32_t* d_trace_id, int n_sessions, int n_traces, int32_t* d_perm, void* stream) {
    if (n_sessions < 0 || n_traces < 1) return fail(ABR_ERR_RANGE, "n_sessions must be >= 0 and n_traces >= 1");
    if (n_sessions == 0) return ABR_OK;
    if (!d_trace_id || !d_perm) return fail(ABR_ERR_INVALID, "trace_id or perm is NULL");
    cudaStream_t st = (cudaStream_t)stream;
    size_t bytes = 0;
    CUDA_TRY(launch_sort_by_trace(d_trace_id, n_sessions, n_traces, d_perm, nullptr, &bytes, st));
    // Scratch: one grow-only device buffer per host thread.  (cudaMallocAsync / cudaFreeAsync around the sort cost 3.6 ms
    // per call: the default pool hands its memory back to the driver at every synchronisation.)  An event orders the
    // buffer's reuse when consecutive calls come in on different streams.
    struct Scratch {
        DeviceBuffer buf; cudaEvent_t last = nullptr;
        ~Scratch() { if (last) cudaEventDestroy(last); }
    };
    thread_local Scratch sc;
    bool fresh = false;
    CUDA_TRY(sc.buf.reserve(bytes, &fresh));
    if (fresh) {   // a new block, on the current device: so is the event
        if (sc.last) { cudaEventDestroy(sc.last); sc.last = nullptr; }
        CUDA_TRY(cudaEventCreateWithFlags(&sc.last, cudaEventDisableTiming));
    } else {
        CUDA_TRY(cudaStreamWaitEvent(st, sc.last, 0));
    }
    CUDA_TRY(launch_sort_by_trace(d_trace_id, n_sessions, n_traces, d_perm, sc.buf.p, &bytes, st));
    CUDA_TRY(cudaEventRecord(sc.last, st));
    return ABR_OK;
}

static int check_capacity(const AbrEnv* env, int n_sessions) {
    if (n_sessions < 0 || n_sessions > env->v.cap) return fail(ABR_ERR_RANGE, "n_sessions %d exceeds capacity %d", n_sessions, env->v.cap);
    return ABR_OK;
}

// A batch of n_sessions fits the session order installed for it, if any.
static int check_order(const AbrEnv* env, int n_sessions) {
    if (env->v.perm && env->n_order != n_sessions)
        return fail(ABR_ERR_STATE, "the installed session order has %d entries, the batch %d (abr_env_set_order)", env->n_order, n_sessions);
    return ABR_OK;
}

// The start of every call on the current batch (an empty batch then makes the call a no-op).
static int check_reset(const AbrEnv* env) {
    if (!env) return fail(ABR_ERR_INVALID, "env is NULL");
    if (!env->was_reset) return fail(ABR_ERR_STATE, "abr_env_reset has not been called");
    return ABR_OK;
}

// What a reset does to the handle: a batch of n_sessions, numbered from session_base, with no steps taken yet.
static void begin_batch(AbrEnv* env, int n_sessions, long long session_base) {
    env->v.n = n_sessions;
    env->v.session_base = session_base;
    env->fresh_partials = 0;
    env->was_reset = true;
    env->step_base = 0;
}

// A built-in policy id the environment can run: RATE reads the history ring, BOLA the log table of positive sizes.
static int check_policy(const AbrEnv* env, int policy) {
    if (policy < ABR_POLICY_FIXED || policy > ABR_POLICY_BOLA) return fail(ABR_ERR_INVALID, "unknown policy %d", policy);
    if (policy == ABR_POLICY_RATE && !env->v.p.track_history)
        return fail(ABR_ERR_STATE, "ABR_POLICY_RATE needs the throughput history: create the environment with track_history = 1");
    if (policy == ABR_POLICY_BOLA && !env->v.pol.bola_v) return fail(ABR_ERR_INVALID, "BOLA needs positive chunk sizes");
    return ABR_OK;
}

int abr_env_set_policy_params(AbrEnv* env, const AbrPolicyParams* params) {
    if (int rc = check_policy_params(params)) return rc;   // host-side only: bad values are reported without a device
    if (!env) return fail(ABR_ERR_INVALID, "env is NULL");
    install_policy_params(env, params);
    return ABR_OK;
}

int abr_env_policy_decide(AbrEnv* env, int policy, int32_t* d_action, void* stream) {
    if (!env) return fail(ABR_ERR_INVALID, "env is NULL");
    if (policy != ABR_POLICY_BBA && policy != ABR_POLICY_RATE && policy != ABR_POLICY_BOLA)
        return fail(ABR_ERR_INVALID, "abr_env_policy_decide takes ABR_POLICY_BBA, _RATE or _BOLA (got %d)", policy);
    if (int rc = check_policy(env, policy)) return rc;
    if (int rc = check_reset(env)) return rc;
    if (env->v.n == 0) return ABR_OK;
    if (!d_action) return fail(ABR_ERR_INVALID, "action is NULL");
    CUDA_TRY(launch_policy_decide(env->v, policy, d_action, (cudaStream_t)stream));
    return ABR_OK;
}

int abr_env_set_order(AbrEnv* env, const int32_t* d_perm, int n_sessions, void* stream) {
    if (!env) return fail(ABR_ERR_INVALID, "env is NULL");
    if (!d_perm) { env->v.perm = nullptr; env->n_order = 0; return ABR_OK; }
    if (int rc = check_capacity(env, n_sessions)) return rc;
    if (!env->d_perm) CUDA_TRY(env->alloc(&env->d_perm, (size_t)env->v.cap));
    CUDA_TRY(cudaMemcpyAsync(env->d_perm, d_perm, sizeof(int32_t) * n_sessions, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    env->v.perm = env->d_perm;
    env->n_order = n_sessions;
    return ABR_OK;
}

int abr_env_reset(AbrEnv* env, const int32_t* d_trace_id, const double* d_start_offset, int n_sessions,
                  long long session_base, void* stream) {
    if (!env || (!d_trace_id && n_sessions > 0)) return fail(ABR_ERR_INVALID, "env or trace_id is NULL");
    if (int rc = check_capacity(env, n_sessions)) return rc;
    if (int rc = check_order(env, n_sessions)) return rc;
    begin_batch(env, n_sessions, session_base);
    CUDA_TRY(launch_reset(env->v, d_trace_id, d_start_offset, env->d_draw_counter, (cudaStream_t)stream));
    return ABR_OK;
}

int abr_env_get_order(AbrEnv* env, int32_t* d_perm, int n_sessions, void* stream) {
    if (!env || !d_perm) return fail(ABR_ERR_INVALID, "env or perm is NULL");
    if (!env->v.perm) return fail(ABR_ERR_STATE, "no session order is installed");
    if (n_sessions != env->n_order) return fail(ABR_ERR_RANGE, "the installed order has %d entries, not %d", env->n_order, n_sessions);
    CUDA_TRY(cudaMemcpyAsync(d_perm, env->d_perm, sizeof(int32_t) * n_sessions, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return ABR_OK;
}

int abr_env_reset_sorted(AbrEnv* env, const int32_t* d_trace_id, const double* d_start_offset, int n_sessions,
                         long long session_base, void* stream) {
    if (!env || (!d_trace_id && n_sessions > 0)) return fail(ABR_ERR_INVALID, "env or trace_id is NULL");
    if (int rc = check_capacity(env, n_sessions)) return rc;
    if (d_trace_id == env->d_trace_id || (d_start_offset && d_start_offset == env->d_offset))
        return fail(ABR_ERR_INVALID, "the inputs alias the environment's own scratch");
    cudaStream_t st = (cudaStream_t)stream;
    if (!env->d_perm) CUDA_TRY(env->alloc(&env->d_perm, (size_t)env->v.cap));
    if (n_sessions > 0) {
        int S = 0, n_blocks = 0;
        sort_shape(n_sessions, env->v.n_traces, &S, &n_blocks);
        if (n_blocks > 0) {
            const size_t cells = (((size_t)env->v.n_traces * n_blocks) + 63) & ~(size_t)63;
            const size_t scan_bytes = sort_scan_tmp_bytes((int)cells);
            bool fresh = false;
            CUDA_TRY(env->sort_hist.reserve(sizeof(int32_t) * cells, &fresh));
            if (fresh) CUDA_TRY(cudaMemset(env->sort_hist.p, 0, env->sort_hist.bytes));   // the sort leaves it zero
            CUDA_TRY(env->sort_scan.reserve(scan_bytes));
            CUDA_TRY(launch_sort_gather(d_trace_id, d_start_offset, n_sessions, env->v.n_traces, S, n_blocks,
                                        env->sort_hist.as<int32_t>(), env->sort_scan.p, scan_bytes,
                                        env->d_perm, env->d_trace_id, env->d_offset, st));
        } else {   // shapes the counting sort does not take: CUB's radix sort, then one gather
            int rc = abr_sort_by_trace(d_trace_id, n_sessions, env->v.n_traces, env->d_perm, stream);
            if (rc) return rc;
            CUDA_TRY(launch_gather(d_trace_id, d_start_offset, env->d_perm, n_sessions, env->d_trace_id, env->d_offset, st));
        }
    }
    env->v.perm = env->d_perm;
    env->n_order = n_sessions;
    return abr_env_reset(env, env->d_trace_id, env->d_offset, n_sessions, session_base, stream);
}

int abr_env_reset_host(AbrEnv* env, const int32_t* h_trace_id, const double* h_start_offset, int n_sessions,
                       long long session_base, void* stream) {
    if (!env || (!h_trace_id && n_sessions > 0)) return fail(ABR_ERR_INVALID, "env or trace_id is NULL");
    if (int rc = check_capacity(env, n_sessions)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaMemcpyAsync(env->d_trace_id, h_trace_id, sizeof(int32_t) * n_sessions, cudaMemcpyHostToDevice, st));
    if (h_start_offset)
        CUDA_TRY(cudaMemcpyAsync(env->d_offset, h_start_offset, sizeof(double) * n_sessions, cudaMemcpyHostToDevice, st));
    return abr_env_reset(env, env->d_trace_id, h_start_offset ? env->d_offset : nullptr, n_sessions, session_base, stream);
}

extern "C++" {
template <typename OT>
static int env_step_any(AbrEnv* env, const int32_t* d_action, const double* d_speed, OT* d_delay, OT* d_sleep,
                        OT* d_buffer, OT* d_rebuf, OT* d_reward, OT* d_latency, OT* d_next_sizes,
                        uint8_t* d_end_of_video, OT* d_throughput, void* stream) {
    if (int rc = check_reset(env)) return rc;
    if (env->v.n == 0) return ABR_OK;
    if (!d_action) return fail(ABR_ERR_INVALID, "action is NULL");
    env->fresh_partials = 0;
    StepOutputs<OT> o;
    o.delay = d_delay; o.sleep = d_sleep; o.buffer = d_buffer; o.rebuf = d_rebuf; o.reward = d_reward;
    o.eov = d_end_of_video; o.latency = d_latency; o.thr = d_throughput; o.next_sizes = d_next_sizes;
    CUDA_TRY(launch_step(env->v, d_action, d_speed, o, (cudaStream_t)stream));
    return ABR_OK;
}
}  // extern "C++"

int abr_env_step_live(AbrEnv* env, const int32_t* d_action, const double* d_speed, double* d_delay, double* d_sleep,
                      double* d_buffer, double* d_rebuf, double* d_reward, double* d_latency, double* d_next_sizes,
                      uint8_t* d_end_of_video, double* d_throughput, void* stream) {
    return env_step_any<double>(env, d_action, d_speed, d_delay, d_sleep, d_buffer, d_rebuf, d_reward, d_latency,
                                d_next_sizes, d_end_of_video, d_throughput, stream);
}

// The checks of the windowed observation's spec and buffer (SPEC §4.5), in their order, and its fields of `pol`.
static int set_obs_window(StepPolicyWindow& pol, const AbrObsWindowSpec* spec, float* d_obs) {
    if (!spec) return fail(ABR_ERR_INVALID, "spec is NULL");
    if (!d_obs) return fail(ABR_ERR_INVALID, "obs is NULL");
    if (spec->window < 1 || spec->window > 32) return fail(ABR_ERR_RANGE, "window must be in [1, 32] (got %d)", spec->window);
    pol.obs = d_obs; pol.window = spec->window;
    pol.w_util = spec->util_scale; pol.w_buffer = spec->buffer_scale; pol.w_thr = spec->throughput_scale;
    pol.w_delay = spec->delay_scale; pol.w_size = spec->size_scale;
    return ABR_OK;
}

extern "C++" {
// The policy-in-the-loop step (SPEC §4.1, §4.5): `name` is the entry point, `observe(pol)` sets its observation
// fields and returns its own checks' result, after the common ones.
template <typename Observe>
static int step_policy_any(AbrEnv* env, const char* name, const float* d_logits, int sample, uint64_t seed,
                           const Observe& observe, int32_t* d_action_out, double* d_reward_sum, double* d_delay,
                           double* d_sleep, double* d_buffer, double* d_rebuf, double* d_reward,
                           uint8_t* d_end_of_video, void* stream) {
    if (int rc = check_reset(env)) return rc;
    if (env->v.p.live) return fail(ABR_ERR_STATE, "%s is not available in live mode (SPEC 7)", name);
    if (env->v.n == 0) return ABR_OK;
    if (!d_logits) return fail(ABR_ERR_INVALID, "logits is NULL");
    StepPolicyWindow pol;
    if (int rc = observe(pol)) return rc;
    pol.logits = d_logits;
    pol.draw = sample ? env->d_draw_counter : nullptr;
    pol.seed_lo = (uint32_t)seed; pol.seed_hi = (uint32_t)(seed >> 32);
    pol.action_out = d_action_out; pol.reward_sum = d_reward_sum;
    env->fresh_partials = 0;
    StepOutputs<double> o;
    o.delay = d_delay; o.sleep = d_sleep; o.buffer = d_buffer; o.rebuf = d_rebuf; o.reward = d_reward;
    o.eov = d_end_of_video;
    CUDA_TRY(launch_step_policy(env->v, pol, o, env->d_draw_counter, (cudaStream_t)stream));
    return ABR_OK;
}
}  // extern "C++"

int abr_env_step_policy(AbrEnv* env, const float* d_logits, int sample, uint64_t seed, const AbrObsSpec* spec,
                        float* d_obs, int32_t* d_action_out, double* d_reward_sum, double* d_delay, double* d_sleep,
                        double* d_buffer, double* d_rebuf, double* d_reward, uint8_t* d_end_of_video, void* stream) {
    auto observe = [&](StepPolicyWindow& pol) {
        pol.obs = d_obs;
        if (spec) {
            pol.s_buffer = spec->buffer_scale; pol.s_thr = spec->throughput_scale;
            pol.s_delay = spec->delay_scale; pol.s_size = spec->size_scale;
        }
        return ABR_OK;
    };
    return step_policy_any(env, "abr_env_step_policy", d_logits, sample, seed, observe, d_action_out, d_reward_sum,
                           d_delay, d_sleep, d_buffer, d_rebuf, d_reward, d_end_of_video, stream);
}

int abr_env_step_policy_window(AbrEnv* env, const float* d_logits, int sample, uint64_t seed,
                               const AbrObsWindowSpec* spec, float* d_obs, int32_t* d_action_out, double* d_reward_sum,
                               double* d_delay, double* d_sleep, double* d_buffer, double* d_rebuf, double* d_reward,
                               uint8_t* d_end_of_video, void* stream) {
    auto observe = [&](StepPolicyWindow& pol) { return set_obs_window(pol, spec, d_obs); };
    return step_policy_any(env, "abr_env_step_policy_window", d_logits, sample, seed, observe, d_action_out,
                           d_reward_sum, d_delay, d_sleep, d_buffer, d_rebuf, d_reward, d_end_of_video, stream);
}

int abr_env_observe_window(AbrEnv* env, const AbrObsWindowSpec* spec, float* d_obs, void* stream) {
    if (int rc = check_reset(env)) return rc;
    if (env->v.p.live) return fail(ABR_ERR_STATE, "abr_env_observe_window is not available in live mode (SPEC 7)");
    if (env->v.n == 0) return ABR_OK;
    StepPolicyWindow pol;
    if (int rc = set_obs_window(pol, spec, d_obs)) return rc;
    CUDA_TRY(launch_observe_window(env->v, pol, (cudaStream_t)stream));
    return ABR_OK;
}

int abr_env_step_f32(AbrEnv* env, const int32_t* d_action, const double* d_speed, float* d_delay, float* d_sleep,
                     float* d_buffer, float* d_rebuf, float* d_reward, float* d_latency, float* d_next_sizes,
                     uint8_t* d_end_of_video, float* d_throughput, void* stream) {
    return env_step_any<float>(env, d_action, d_speed, d_delay, d_sleep, d_buffer, d_rebuf, d_reward, d_latency,
                               d_next_sizes, d_end_of_video, d_throughput, stream);
}

int abr_env_step(AbrEnv* env, const int32_t* d_action, double* d_delay, double* d_sleep, double* d_buffer,
                 double* d_rebuf, double* d_reward, double* d_next_sizes, uint8_t* d_end_of_video, double* d_throughput,
                 void* stream) {
    return abr_env_step_live(env, d_action, nullptr, d_delay, d_sleep, d_buffer, d_rebuf, d_reward, nullptr,
                             d_next_sizes, d_end_of_video, d_throughput, stream);
}

int abr_env_qoe_cost(AbrEnv* env, double* d_out, void* stream) {
    if (!env || !d_out) return fail(ABR_ERR_INVALID, "env or out is NULL");
    CUDA_TRY(launch_qoe_cost(env->v, d_out, (cudaStream_t)stream));
    return ABR_OK;
}

extern "C++" {
// A fused episode of the current batch, whose other arguments have passed the caller's checks.
template <typename OT>
static int episode(AbrEnv* env, int policy, uint64_t seed, int steps, const int32_t* d_actions_in, const double* d_speed,
                   const StepOutputs<OT>& o, cudaStream_t st, const RolloutFused& fused = RolloutFused{}) {
    // the kernel indexes the [steps][N] outputs with 32 bits (4 Gi elements of one array are 32 GB)
    if ((unsigned long long)steps * (unsigned long long)env->v.n > 0xffffffffull)
        return fail(ABR_ERR_RANGE, "steps * sessions = %llu exceeds 2^32 - 1: split the episode into several calls",
                    (unsigned long long)steps * (unsigned long long)env->v.n);
    CUDA_TRY(launch_rollout(env->v, policy, seed, steps, env->step_base, d_actions_in, d_speed, o, env->d_stats_partials,
                            fused, st));
    env->step_base += (uint32_t)steps;
    env->fresh_partials = steps > 0 ? rollout_num_blocks(env->v.n) : 0;
    return ABR_OK;
}

template <typename OT>
static int env_rollout_any(AbrEnv* env, int policy, uint64_t seed, int steps, const int32_t* d_actions_in,
                           const double* d_speed, OT* d_delay, OT* d_sleep, OT* d_buffer, OT* d_rebuf, OT* d_reward,
                           OT* d_latency, uint8_t* d_end_of_video, int32_t* d_actions_out, void* stream) {
    if (int rc = check_reset(env)) return rc;
    if (env->v.n == 0) return ABR_OK;
    if (steps < 0) return fail(ABR_ERR_RANGE, "steps must be >= 0");
    if (int rc_p = check_policy(env, policy)) return rc_p;
    if (policy == ABR_POLICY_FIXED && !d_actions_in) return fail(ABR_ERR_INVALID, "ABR_POLICY_FIXED needs d_actions_in");
    if (!env->v.p.live && (d_speed || d_latency))
        return fail(ABR_ERR_STATE, "speed / latency belong to live mode (SPEC 7): create the environment with live = 1");
    StepOutputs<OT> o;
    o.delay = d_delay; o.sleep = d_sleep; o.buffer = d_buffer; o.rebuf = d_rebuf; o.reward = d_reward;
    o.eov = d_end_of_video; o.actions = d_actions_out; o.latency = d_latency;
    return episode(env, policy, seed, steps, d_actions_in, d_speed, o, (cudaStream_t)stream);
}
}  // extern "C++"

int abr_env_rollout_fused_live(AbrEnv* env, int policy, uint64_t seed, int steps, const int32_t* d_actions_in,
                               const double* d_speed, double* d_delay, double* d_sleep, double* d_buffer,
                               double* d_rebuf, double* d_reward, double* d_latency, uint8_t* d_end_of_video,
                               int32_t* d_actions_out, void* stream) {
    return env_rollout_any<double>(env, policy, seed, steps, d_actions_in, d_speed, d_delay, d_sleep, d_buffer,
                                   d_rebuf, d_reward, d_latency, d_end_of_video, d_actions_out, stream);
}

int abr_env_rollout_fused_f32(AbrEnv* env, int policy, uint64_t seed, int steps, const int32_t* d_actions_in,
                              const double* d_speed, float* d_delay, float* d_sleep, float* d_buffer, float* d_rebuf,
                              float* d_reward, float* d_latency, uint8_t* d_end_of_video, int32_t* d_actions_out,
                              void* stream) {
    return env_rollout_any<float>(env, policy, seed, steps, d_actions_in, d_speed, d_delay, d_sleep, d_buffer,
                                  d_rebuf, d_reward, d_latency, d_end_of_video, d_actions_out, stream);
}

int abr_env_rollout_fused(AbrEnv* env, int policy, uint64_t seed, int steps, const int32_t* d_actions_in,
                          double* d_delay, double* d_sleep, double* d_buffer, double* d_rebuf, double* d_reward,
                          uint8_t* d_end_of_video, int32_t* d_actions_out, void* stream) {
    return abr_env_rollout_fused_live(env, policy, seed, steps, d_actions_in, nullptr, d_delay, d_sleep, d_buffer,
                                      d_rebuf, d_reward, nullptr, d_end_of_video, d_actions_out, stream);
}

static int check_mpc_shape(int A, int H) {
    if (H < 1 || H > 8) return fail(ABR_ERR_RANGE, "horizon must be in [1, 8] (got %d)", H);
    if (A < 1 || A > 16) return fail(ABR_ERR_RANGE, "A must be in [1, 16]");
    double combos = 1;
    for (int i = 0; i < H; ++i) combos *= A;
    if (combos > 2147483647.0) return fail(ABR_ERR_RANGE, "A^H = %g sequences exceed the 2^31-1 index range", combos);
    return ABR_OK;
}

int abr_env_mpc_decide(AbrEnv* env, int horizon, int mode, int32_t* d_action, double* d_best_j, void* stream) {
    if (int rc = check_reset(env)) return rc;
    if (env->v.n == 0) return ABR_OK;
    if (!d_action) return fail(ABR_ERR_INVALID, "action is NULL");
    const bool exhaustive = (mode & ABR_MPC_MODE_EXHAUSTIVE) != 0;
    mode &= ~ABR_MPC_MODE_EXHAUSTIVE;
    if (mode != ABR_MPC_REF && mode != ABR_MPC_ROBUST) return fail(ABR_ERR_INVALID, "unknown MPC mode %d", mode);
    if (!env->v.p.track_history)
        return fail(ABR_ERR_STATE, "abr_env_mpc_decide needs the throughput history: create the environment with track_history = 1");
    int rc = check_mpc_shape(env->v.A, horizon);
    if (rc) return rc;
    const EnvView& v = env->v;
    MpcArgs a{};
    a.sizes = v.sizes; a.util = v.util; a.V = v.V; a.A = v.A; a.p = v.p; a.N = v.n;
    a.chunk_idx = v.chunk; a.prev_q = v.last_q; a.buffer = v.buffer; a.done = v.p.auto_reset ? nullptr : v.done;
    a.bw_hist = v.bw_hist; a.hist_len = v.hist_len; a.K = v.K;
    a.hist_session_stride = 1; a.hist_slot_stride = v.cap;     // env rings are [K][cap]
    a.last_pred = v.last_pred; a.err_ring = v.err_ring; a.err_len = v.err_len;
    a.H = horizon; a.mode = mode; a.flags = ABR_MPC_TRUNCATE | ABR_MPC_EMPTY_DEFAULT | (exhaustive ? ABR_MPC_EXHAUSTIVE : 0);
    a.action = d_action; a.best_j = d_best_j; a.best_seq = nullptr; a.preds = nullptr;
    a.error_count64 = v.errors; a.error_count32 = nullptr;
    CUDA_TRY(launch_mpc(a, (cudaStream_t)stream));
    return ABR_OK;
}

int abr_env_mpc_decide_pred(AbrEnv* env, int horizon, int flags, const double* d_pred, int32_t* d_action,
                            double* d_best_j, int32_t* d_best_seq, void* stream) {
    if (int rc = check_reset(env)) return rc;
    if (env->v.n == 0) return ABR_OK;
    if (!d_action) return fail(ABR_ERR_INVALID, "action is NULL");
    if (!d_pred) return fail(ABR_ERR_INVALID, "pred is NULL");
    if (flags != 0 && flags != ABR_MPC_EXHAUSTIVE)
        return fail(ABR_ERR_INVALID, "flags must be 0 or ABR_MPC_EXHAUSTIVE (got %d)", flags);
    if (int rc = check_mpc_shape(env->v.A, horizon)) return rc;
    const EnvView& v = env->v;
    MpcArgs a{};   // no history ring and no robust state: the kernel reads neither (SPEC §5.6)
    a.sizes = v.sizes; a.util = v.util; a.V = v.V; a.A = v.A; a.p = v.p; a.N = v.n;
    a.chunk_idx = v.chunk; a.prev_q = v.last_q; a.buffer = v.buffer; a.done = v.p.auto_reset ? nullptr : v.done;
    a.K = v.K;
    a.H = horizon; a.mode = ABR_MPC_ROBUST; a.flags = flags;
    a.action = d_action; a.best_j = d_best_j; a.best_seq = d_best_seq;
    a.error_count64 = v.errors;
    a.pred = d_pred;
    CUDA_TRY(launch_mpc(a, (cudaStream_t)stream));
    return ABR_OK;
}

int abr_env_mpc_decide_scen(AbrEnv* env, int horizon, int n_scen, int objective, int flags, const double* d_pred,
                            const double* d_weight, int32_t* d_action, double* d_best_j, int32_t* d_best_seq,
                            void* stream) {
    if (int rc = check_reset(env)) return rc;
    if (env->v.n == 0) return ABR_OK;
    if (!d_action) return fail(ABR_ERR_INVALID, "action is NULL");
    if (!d_pred) return fail(ABR_ERR_INVALID, "pred is NULL");
    if (objective != ABR_MPC_SCEN_MEAN && objective != ABR_MPC_SCEN_WORST)
        return fail(ABR_ERR_INVALID, "objective must be ABR_MPC_SCEN_MEAN or ABR_MPC_SCEN_WORST (got %d)", objective);
    if (d_weight && objective == ABR_MPC_SCEN_WORST)
        return fail(ABR_ERR_INVALID, "weights apply to ABR_MPC_SCEN_MEAN only");
    if (flags != 0 && flags != ABR_MPC_EXHAUSTIVE)
        return fail(ABR_ERR_INVALID, "flags must be 0 or ABR_MPC_EXHAUSTIVE (got %d)", flags);
    if (int rc = check_mpc_shape(env->v.A, horizon)) return rc;
    if (n_scen < 1 || n_scen > ABR_MPC_SCEN_MAX)
        return fail(ABR_ERR_RANGE, "n_scen must be in [1, %d] (got %d)", ABR_MPC_SCEN_MAX, n_scen);
    const EnvView& v = env->v;
    MpcScenArgs a{};   // no history ring and no robust state: the kernel reads neither (SPEC 5.7)
    a.sizes = v.sizes; a.util = v.util; a.V = v.V; a.A = v.A; a.p = v.p; a.N = v.n;
    a.chunk_idx = v.chunk; a.prev_q = v.last_q; a.buffer = v.buffer; a.done = v.p.auto_reset ? nullptr : v.done;
    a.H = horizon; a.K = n_scen; a.objective = objective; a.flags = flags;
    a.pred = d_pred; a.weight = d_weight;
    a.action = d_action; a.best_j = d_best_j; a.best_seq = d_best_seq;
    a.error_count64 = v.errors;
    CUDA_TRY(launch_mpc_scen(a, (cudaStream_t)stream));
    return ABR_OK;
}

int abr_env_lookahead_decide(AbrEnv* env, int horizon, int32_t* d_action, double* d_best_value, int32_t* d_best_seq,
                             void* stream) {
    if (int rc = check_reset(env)) return rc;
    if (env->v.p.live) return fail(ABR_ERR_STATE, "abr_env_lookahead_decide is not available in live mode (SPEC 7)");
    if (env->v.n == 0) return ABR_OK;
    if (!d_action) return fail(ABR_ERR_INVALID, "action is NULL");
    if (horizon < 1 || horizon > 8) return fail(ABR_ERR_RANGE, "horizon must be in [1, 8] (got %d)", horizon);
    double combos = 1;
    for (int i = 0; i < horizon; ++i) combos *= env->v.A;
    if (combos > 1048576.0)
        return fail(ABR_ERR_RANGE, "A^horizon = %g sequences exceed the lookahead limit of 2^20 = 1048576", combos);
    CUDA_TRY(launch_lookahead(env->v, horizon, d_action, d_best_value, d_best_seq, (cudaStream_t)stream));
    return ABR_OK;
}

int abr_stats_partial(AbrEnv* env, double* d_out, void* stream) {
    if (!env || !d_out) return fail(ABR_ERR_INVALID, "env or out is NULL");
    const bool fresh = env->fresh_partials > 0;
    const int np = fresh ? env->fresh_partials : stats_num_partials(env->v.n);
    CUDA_TRY(launch_stats(env->v, env->d_stats_partials, np, fresh, d_out, env->stats_scratch, (cudaStream_t)stream));
    return ABR_OK;
}

int abr_env_state_ptr(AbrEnv* env, int field, void** d_ptr) {
    if (!env || !d_ptr) return fail(ABR_ERR_INVALID, "env or d_ptr is NULL");
    const EnvView& v = env->v;
    switch (field) {
        case ABR_F_SEG: *d_ptr = v.seg; break;
        case ABR_F_CHUNK: *d_ptr = v.chunk; break;
        case ABR_F_LAST_Q: *d_ptr = v.last_q; break;
        case ABR_F_TRACE_ID: *d_ptr = v.trace_id; break;
        case ABR_F_HIST_LEN: *d_ptr = v.hist_len; break;
        case ABR_F_DONE: *d_ptr = v.done; break;
        case ABR_F_ERR_LEN: *d_ptr = v.err_len; break;
        case ABR_F_PHASE: *d_ptr = v.phi; break;
        case ABR_F_POS: *d_ptr = v.pos; break;
        case ABR_F_BUFFER: *d_ptr = v.buffer; break;
        case ABR_F_BW_HIST: *d_ptr = v.bw_hist; break;
        case ABR_F_LAST_PRED: *d_ptr = v.last_pred; break;
        case ABR_F_ERR_RING: *d_ptr = v.err_ring; break;
        case ABR_F_ACC: *d_ptr = v.acc; break;
        case ABR_F_T_NOW: *d_ptr = v.t_now; break;
        case ABR_F_PLAY_TIME: *d_ptr = v.play_time; break;
        case ABR_F_STARTED: *d_ptr = v.started; break;
        case ABR_F_PLAY_ID: *d_ptr = v.play_id; break;
        case ABR_F_PLAY_LEN: *d_ptr = v.play_len; break;
        case ABR_F_SIZES: *d_ptr = (void*)v.sizes; break;
        case ABR_F_UTILITY: *d_ptr = (void*)v.util; break;
        case ABR_F_TRACE_BW: *d_ptr = (void*)v.trace_bw; break;
        case ABR_F_ORDER:
            if (!v.perm) return fail(ABR_ERR_STATE, "no session order is installed");
            *d_ptr = (void*)v.perm; break;
        default: return fail(ABR_ERR_INVALID, "unknown state field %d", field);
    }
    return ABR_OK;
}

int abr_env_error_count(AbrEnv* env, long long* out, void* stream) {
    if (!env || !out) return fail(ABR_ERR_INVALID, "env or out is NULL");
    unsigned long long h = 0;
    CUDA_TRY(cudaMemcpyAsync(&h, env->v.errors, sizeof(h), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    *out = (long long)h;
    return ABR_OK;
}

// abr_env_run and abr_env_run_host on device pointers, after their checks: with sessions and steps, one episode kernel
// that resets the sessions itself (no state round trip through HBM) and writes the session cost and the statistics;
// otherwise the reset, the cost and the statistics of the reset state.
static int run_batch(AbrEnv* env, int policy, uint64_t seed, int steps, const int32_t* d_trace_id,
                     const double* d_start_offset, int n_sessions, long long session_base, const int32_t* d_actions_in,
                     const StepOutputs<double>& o, double* d_qoe_cost, double* d_stats, cudaStream_t st) {
    begin_batch(env, n_sessions, session_base);
    if (n_sessions > 0 && steps > 0) {
        RolloutFused fused;
        fused.in_trace_id = d_trace_id; fused.in_offset = d_start_offset; fused.out_cost = d_qoe_cost;
        fused.out_stats = d_stats; fused.scratch = env->stats_scratch;   // statistics by the kernel's own blocks
        return episode(env, policy, seed, steps, d_actions_in, nullptr, o, st, fused);
    }
    CUDA_TRY(launch_reset(env->v, d_trace_id, d_start_offset, env->d_draw_counter, st));
    if (d_qoe_cost) CUDA_TRY(launch_qoe_cost(env->v, d_qoe_cost, st));
    return d_stats ? abr_stats_partial(env, d_stats, st) : ABR_OK;
}

int abr_env_run(AbrEnv* env, int policy, uint64_t seed, int steps, const int32_t* d_trace_id,
                const double* d_start_offset, int n_sessions, long long session_base, const int32_t* d_actions_in,
                double* d_delay, double* d_sleep, double* d_buffer, double* d_rebuf, double* d_reward,
                uint8_t* d_end_of_video, int32_t* d_actions_out, double* d_qoe_cost, double* d_stats, void* stream) {
    if (!env || (!d_trace_id && n_sessions > 0)) return fail(ABR_ERR_INVALID, "env or trace_id is NULL");
    if (int rc = check_capacity(env, n_sessions)) return rc;
    if (steps < 0) return fail(ABR_ERR_RANGE, "steps must be >= 0");
    if (int rc = check_policy(env, policy)) return rc;
    if (policy == ABR_POLICY_FIXED && !d_actions_in && n_sessions > 0 && steps > 0)
        return fail(ABR_ERR_INVALID, "ABR_POLICY_FIXED needs d_actions_in");
    if (int rc = check_order(env, n_sessions)) return rc;
    StepOutputs<double> o;
    o.delay = d_delay; o.sleep = d_sleep; o.buffer = d_buffer; o.rebuf = d_rebuf; o.reward = d_reward;
    o.eov = d_end_of_video; o.actions = d_actions_out;
    return run_batch(env, policy, seed, steps, d_trace_id, d_start_offset, n_sessions, session_base, d_actions_in, o,
                     d_qoe_cost, d_stats, (cudaStream_t)stream);
}

// Zero-copy: a host pointer inside page-locked memory (cudaHostAlloc / cudaHostRegister, e.g. a pinned torch tensor)
// has a device alias under unified addressing; the kernels then read the inputs and write the results over PCIe
// themselves, which removes the copy launches and overlaps the transfers with the kernels' other work.  Returns
// nullptr for pageable memory (the staged cudaMemcpyAsync path is used).
static void* device_alias(const void* h) {
    if (!h) return nullptr;
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, h) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return a.type == cudaMemoryTypeHost ? a.devicePointer : nullptr;
}

int abr_env_run_host(AbrEnv* env, int policy, uint64_t seed, int steps, const int32_t* h_trace_id,
                     const double* h_start_offset, int n_sessions, long long session_base, const int32_t* h_actions_in,
                     double* h_acc, double* h_stats, double* h_reward_traj, double* h_qoe_cost, void* stream) {
    if (!env) return fail(ABR_ERR_INVALID, "env is NULL");
    if (steps < 0) return fail(ABR_ERR_RANGE, "steps must be >= 0");
    if (!h_trace_id && n_sessions > 0) return fail(ABR_ERR_INVALID, "env or trace_id is NULL");
    if (int rc = check_capacity(env, n_sessions)) return rc;
    if (int rc = check_policy(env, policy)) return rc;
    if (policy == ABR_POLICY_FIXED && !h_actions_in) return fail(ABR_ERR_INVALID, "ABR_POLICY_FIXED needs h_actions_in");
    if (int rc = check_order(env, n_sessions)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    // inputs: device aliases of page-locked buffers (read over PCIe by the kernels), else copies into the scratch
    const int32_t* tid = (const int32_t*)device_alias(h_trace_id);
    if (!tid) {
        if (n_sessions > 0)
            CUDA_TRY(cudaMemcpyAsync(env->d_trace_id, h_trace_id, sizeof(int32_t) * n_sessions, cudaMemcpyHostToDevice, st));
        tid = env->d_trace_id;
    }
    const double* off = (const double*)device_alias(h_start_offset);
    if (h_start_offset && !off) {
        CUDA_TRY(cudaMemcpyAsync(env->d_offset, h_start_offset, sizeof(double) * n_sessions, cudaMemcpyHostToDevice, st));
        off = env->d_offset;
    }
    const size_t traj = (size_t)steps * n_sessions;
    const int32_t* d_actions = nullptr;
    if (policy == ABR_POLICY_FIXED) {
        CUDA_TRY(env->actions.reserve(sizeof(int32_t) * traj));
        d_actions = env->actions.as<int32_t>();
        CUDA_TRY(cudaMemcpyAsync(env->actions.p, h_actions_in, sizeof(int32_t) * traj, cudaMemcpyHostToDevice, st));
    }
    StepOutputs<double> o;
    if (h_reward_traj) {
        CUDA_TRY(env->reward_traj.reserve(sizeof(double) * traj));
        o.reward = env->reward_traj.as<double>();
    }
    // outputs: page-locked ones are written by the kernels through their aliases; pageable statistics go through
    // d_stats_out, a pageable cost through d_offset (free again once the sessions are reset) by a launch of its own
    double* z_cost = (double*)device_alias(h_qoe_cost);
    double* z_stats = (double*)device_alias(h_stats);
    if (int rc = run_batch(env, policy, seed, steps, tid, off, n_sessions, session_base, d_actions, o, z_cost,
                           h_stats && !z_stats ? env->d_stats_out : z_stats, st))
        return rc;
    if (h_stats && !z_stats)
        CUDA_TRY(cudaMemcpyAsync(h_stats, env->d_stats_out, sizeof(double) * ABR_NUM_STATS, cudaMemcpyDeviceToHost, st));
    if (h_acc) {
        // acc rows are strided by the capacity on the device; the host table is dense [ABR_NUM_ACC][N]
        CUDA_TRY(cudaMemcpy2DAsync(h_acc, sizeof(double) * n_sessions, env->v.acc, sizeof(double) * env->v.cap,
                                   sizeof(double) * n_sessions, ABR_NUM_ACC, cudaMemcpyDeviceToHost, st));
    }
    if (h_reward_traj)
        CUDA_TRY(cudaMemcpyAsync(h_reward_traj, o.reward, sizeof(double) * traj, cudaMemcpyDeviceToHost, st));
    if (h_qoe_cost && !z_cost) {
        CUDA_TRY(launch_qoe_cost(env->v, env->d_offset, st));
        CUDA_TRY(cudaMemcpyAsync(h_qoe_cost, env->d_offset, sizeof(double) * n_sessions, cudaMemcpyDeviceToHost, st));
    }
    CUDA_TRY(cudaStreamSynchronize(st));
    return ABR_OK;
}

// The standalone decision of abr_mpc_decide*: checks the arguments `a` names, completes it and launches.
static int mpc_decide(MpcArgs a, const AbrParams* params, cudaStream_t st) {
    if (!a.sizes || !a.util || !a.chunk_idx || !a.prev_q || !a.buffer || !a.bw_hist || !a.hist_len || !a.action)
        return fail(ABR_ERR_INVALID, "a required pointer is NULL");
    if (!params) return fail(ABR_ERR_INVALID, "params is NULL");
    if (a.N < 0 || a.V < 1) return fail(ABR_ERR_RANGE, "N must be >= 0 and V >= 1");
    if (a.K < 1) return fail(ABR_ERR_RANGE, "K must be >= 1");
    if (a.mode != ABR_MPC_REF && a.mode != ABR_MPC_ROBUST) return fail(ABR_ERR_INVALID, "unknown MPC mode %d", a.mode);
    if ((a.flags & ABR_MPC_PRED_SES) && a.mode != ABR_MPC_REF)
        return fail(ABR_ERR_INVALID, "ABR_MPC_PRED_SES (mpc.py:72-79) replaces the predictor of mode 0; the robust mode defines its own");
    if ((a.last_pred || a.err_ring || a.err_len) && !(a.last_pred && a.err_ring && a.err_len))
        return fail(ABR_ERR_INVALID, "last_pred, err_ring and err_len must be given together");
    if (a.n_ts < 1 || a.n_ts > 4096) return fail(ABR_ERR_RANGE, "n_ts must be in [1, 4096] (got %d)", a.n_ts);
    if (a.n_ts > 1 && !(a.ts_step > 0.0 && std::isfinite(a.ts_step))) return fail(ABR_ERR_RANGE, "ts_step must be finite and > 0");
    if (a.n_ts > 1 && !std::isfinite(params->startup_penalty)) return fail(ABR_ERR_INVALID, "startup_penalty must be finite");
    if (int rc = check_mpc_shape(a.A, a.H)) return rc;
    a.p = *params;
    a.hist_session_stride = a.K; a.hist_slot_stride = 1;        // standalone rings are [N][K]
    CUDA_TRY(launch_mpc(a, st));
    return ABR_OK;
}

int abr_mpc_decide(const double* d_sizes, const double* d_utility, int V, int A, const AbrParams* params, int N,
                   const int32_t* d_chunk_idx, const int32_t* d_prev_q, const double* d_buffer, const double* d_bw_hist,
                   const int32_t* d_hist_len, int K, double* d_last_pred, double* d_err_ring, int32_t* d_err_len,
                   int horizon, int mode, int flags, int32_t* d_action, double* d_best_j, int32_t* d_best_seq,
                   double* d_preds, int32_t* d_error_count, void* stream) {
    MpcArgs a{};
    a.sizes = d_sizes; a.util = d_utility; a.V = V; a.A = A; a.N = N; a.K = K; a.H = horizon; a.mode = mode; a.flags = flags;
    a.chunk_idx = d_chunk_idx; a.prev_q = d_prev_q; a.buffer = d_buffer; a.bw_hist = d_bw_hist; a.hist_len = d_hist_len;
    a.last_pred = d_last_pred; a.err_ring = d_err_ring; a.err_len = d_err_len;
    a.action = d_action; a.best_j = d_best_j; a.best_seq = d_best_seq; a.preds = d_preds; a.error_count32 = d_error_count;
    return mpc_decide(a, params, (cudaStream_t)stream);
}

int abr_mpc_decide_startup(const double* d_sizes, const double* d_utility, int V, int A, const AbrParams* params, int N,
                           const int32_t* d_chunk_idx, const int32_t* d_prev_q, const double* d_buffer,
                           const double* d_bw_hist, const int32_t* d_hist_len, int K, double* d_last_pred,
                           double* d_err_ring, int32_t* d_err_len, int horizon, int mode, int flags,
                           const uint8_t* d_startup, int n_ts, double ts_step, int32_t* d_action,
                           double* d_startup_delay, double* d_best_j, int32_t* d_best_seq, double* d_preds,
                           int32_t* d_error_count, void* stream) {
    if (!d_startup_delay) return fail(ABR_ERR_INVALID, "startup_delay is NULL");
    MpcArgs a{};
    a.sizes = d_sizes; a.util = d_utility; a.V = V; a.A = A; a.N = N; a.K = K; a.H = horizon; a.mode = mode; a.flags = flags;
    a.chunk_idx = d_chunk_idx; a.prev_q = d_prev_q; a.buffer = d_buffer; a.bw_hist = d_bw_hist; a.hist_len = d_hist_len;
    a.last_pred = d_last_pred; a.err_ring = d_err_ring; a.err_len = d_err_len;
    a.action = d_action; a.best_j = d_best_j; a.best_seq = d_best_seq; a.preds = d_preds; a.error_count32 = d_error_count;
    a.startup = d_startup; a.n_ts = n_ts; a.ts_step = ts_step; a.startup_delay = d_startup_delay;
    return mpc_decide(a, params, (cudaStream_t)stream);
}

// The host tables and parameters of abr_mpc_decide*_host and abr_mpc_score_host.
static int check_host_tables(const double* h_sizes, const double* h_bitrates, int V, int A, const AbrParams* params) {
    if (int rc = check_tables(h_sizes, h_bitrates, V, A)) return rc;
    return params ? ABR_OK : fail(ABR_ERR_INVALID, "params is NULL");
}

// ---- host-buffer decisions: one staging arena per host thread (grow-only, released at thread exit), so that a
//      decision is one host->device copy, one kernel and one device->host copy — no allocation on the call path ----
namespace {
struct HostArena {
    DeviceBuffer dev;
    char* pin = nullptr;   // as large as dev
    ~HostArena() { if (pin) cudaFreeHost(pin); }
    cudaError_t reserve(size_t bytes) {
        bool fresh = false;
        cudaError_t e = dev.reserve(bytes < (64u << 10) ? (64u << 10) : bytes, &fresh);
        if (e != cudaSuccess || (pin && !fresh)) return e;
        if (pin) cudaFreeHost(pin);
        e = cudaHostAlloc((void**)&pin, dev.bytes, cudaHostAllocDefault);
        if (e != cudaSuccess) pin = nullptr;
        return e;
    }
};
thread_local HostArena t_arena;
inline size_t align16(size_t x) { return (x + 15) & ~(size_t)15; }
extern "C++" template <typename T>
void point(T*& field, char* base, size_t off) { field = reinterpret_cast<T*>(base + off); }
}  // namespace

// `a` names the caller's host buffers (sizes: the size table; util: unused, the utilities are computed from
// h_bitrates).  They are packed into the arena and copied to the device in one piece, `a` is re-pointed at the device
// copies for mpc_decide, and the outputs come back the same way.  A partial robust state counts as none.
static int mpc_decide_host(MpcArgs a, const double* h_bitrates, const AbrParams* params) {
    if (!a.chunk_idx || !a.prev_q || !a.buffer || !a.bw_hist || !a.hist_len || !a.action)
        return fail(ABR_ERR_INVALID, "a required pointer is NULL");
    if (int rc = check_host_tables(a.sizes, h_bitrates, a.V, a.A, params)) return rc;
    if (a.N < 0 || a.K < 1) return fail(ABR_ERR_RANGE, "N must be >= 0 and K >= 1");
    if (int rc = check_mpc_shape(a.A, a.H)) return rc;
    if (int rc = require_device()) return rc;
    std::vector<double> util;
    utility_table(h_bitrates, a.V, a.A, params, util);
    a.util = util.data();
    if (!(a.last_pred && a.err_ring && a.err_len)) { a.last_pred = a.err_ring = nullptr; a.err_len = nullptr; }
    const MpcArgs h = a;
    const size_t N = (size_t)a.N, n = N > 0 ? N : 1, K = (size_t)a.K, H = (size_t)a.H, VA = (size_t)a.V * a.A;
    // arena layout: [inputs, copied host->device in one piece | outputs, copied back in one piece]
    size_t off = 0;
    auto take = [&off](size_t bytes) { const size_t o = off; off = align16(off + bytes); return o; };
    const size_t o_sizes = take(8 * VA), o_util = take(8 * VA), o_buffer = take(8 * n), o_hist = take(8 * n * K);
    const size_t o_chunk = take(4 * n), o_pq = take(4 * n), o_hl = take(4 * n), o_su = take(n);
    const size_t o_out = off;          // robust state is both input and output: it sits at the start of the output part
    const size_t o_lp = take(8 * n), o_er = take(8 * n * K), o_el = take(4 * n), o_ec = take(16);
    const size_t in_bytes = off;       // inputs end here (the error counter is zeroed on the host side of the copy)
    const size_t o_act = take(4 * n), o_ts = take(8 * n), o_bj = take(8 * n), o_seq = take(4 * n * H), o_pr = take(8 * n * H);
    const size_t total = off;
    CUDA_TRY(t_arena.reserve(total));
    char* hp = t_arena.pin;
    char* dp = t_arena.dev.as<char>();
    auto in = [&](auto*& field, size_t o, size_t bytes) {   // an input: packed, then read from its device copy
        if (!field) return;
        memcpy(hp + o, field, bytes);
        point(field, dp, o);
    };
    in(a.sizes, o_sizes, 8 * VA); in(a.util, o_util, 8 * VA); in(a.buffer, o_buffer, 8 * N); in(a.bw_hist, o_hist, 8 * N * K);
    in(a.chunk_idx, o_chunk, 4 * N); in(a.prev_q, o_pq, 4 * N); in(a.hist_len, o_hl, 4 * N); in(a.startup, o_su, N);
    in(a.last_pred, o_lp, 8 * N); in(a.err_ring, o_er, 8 * N * K); in(a.err_len, o_el, 4 * N);
    memset(hp + o_ec, 0, 16);
    point(a.action, dp, o_act); point(a.startup_delay, dp, o_ts); point(a.best_j, dp, o_bj); point(a.best_seq, dp, o_seq);
    point(a.preds, dp, o_pr); point(a.error_count32, dp, o_ec);
    cudaStream_t st = 0;
    CUDA_TRY(cudaMemcpyAsync(dp, hp, in_bytes, cudaMemcpyHostToDevice, st));
    if (int rc = mpc_decide(a, params, st)) return rc;
    CUDA_TRY(cudaMemcpyAsync(hp + o_out, dp + o_out, total - o_out, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    auto out = [hp](void* dst, size_t o, size_t bytes) { if (dst) memcpy(dst, hp + o, bytes); };
    out(h.action, o_act, 4 * N); out(h.startup_delay, o_ts, 8 * N); out(h.best_j, o_bj, 8 * N);
    out(h.best_seq, o_seq, 4 * N * H); out(h.preds, o_pr, 8 * N * H); out(h.error_count32, o_ec, 4);
    out(h.last_pred, o_lp, 8 * N); out(h.err_ring, o_er, 8 * N * K); out(h.err_len, o_el, 4 * N);
    return ABR_OK;
}

int abr_mpc_decide_host(const double* h_sizes, const double* h_bitrates, int V, int A, const AbrParams* params, int N,
                        const int32_t* h_chunk_idx, const int32_t* h_prev_q, const double* h_buffer,
                        const double* h_bw_hist, const int32_t* h_hist_len, int K, double* h_last_pred,
                        double* h_err_ring, int32_t* h_err_len, int horizon, int mode, int flags, int32_t* h_action,
                        double* h_best_j, int32_t* h_best_seq, double* h_preds, int32_t* h_error_count) {
    MpcArgs a{};
    a.sizes = h_sizes; a.V = V; a.A = A; a.N = N; a.K = K; a.H = horizon; a.mode = mode; a.flags = flags;
    a.chunk_idx = h_chunk_idx; a.prev_q = h_prev_q; a.buffer = h_buffer; a.bw_hist = h_bw_hist; a.hist_len = h_hist_len;
    a.last_pred = h_last_pred; a.err_ring = h_err_ring; a.err_len = h_err_len;
    a.action = h_action; a.best_j = h_best_j; a.best_seq = h_best_seq; a.preds = h_preds; a.error_count32 = h_error_count;
    return mpc_decide_host(a, h_bitrates, params);
}

int abr_mpc_decide_startup_host(const double* h_sizes, const double* h_bitrates, int V, int A, const AbrParams* params,
                                int N, const int32_t* h_chunk_idx, const int32_t* h_prev_q, const double* h_buffer,
                                const double* h_bw_hist, const int32_t* h_hist_len, int K, double* h_last_pred,
                                double* h_err_ring, int32_t* h_err_len, int horizon, int mode, int flags,
                                const uint8_t* h_startup, int n_ts, double ts_step, int32_t* h_action,
                                double* h_startup_delay, double* h_best_j, int32_t* h_best_seq, double* h_preds,
                                int32_t* h_error_count) {
    if (!h_startup_delay) return fail(ABR_ERR_INVALID, "startup_delay is NULL");
    MpcArgs a{};
    a.sizes = h_sizes; a.V = V; a.A = A; a.N = N; a.K = K; a.H = horizon; a.mode = mode; a.flags = flags;
    a.chunk_idx = h_chunk_idx; a.prev_q = h_prev_q; a.buffer = h_buffer; a.bw_hist = h_bw_hist; a.hist_len = h_hist_len;
    a.last_pred = h_last_pred; a.err_ring = h_err_ring; a.err_len = h_err_len;
    a.action = h_action; a.best_j = h_best_j; a.best_seq = h_best_seq; a.preds = h_preds; a.error_count32 = h_error_count;
    a.startup = h_startup; a.n_ts = n_ts; a.ts_step = ts_step; a.startup_delay = h_startup_delay;
    return mpc_decide_host(a, h_bitrates, params);
}

int abr_mpc_score_host(const double* h_sizes, const double* h_bitrates, int V, int A, const AbrParams* params,
                       int chunk_idx, int prev_q, double buffer, const double* h_history, int n_history, int horizon,
                       int mode, double max_err, const int32_t* h_sequences, int M, double* h_scores) {
    if (!h_history || !h_sequences || !h_scores) return fail(ABR_ERR_INVALID, "a required pointer is NULL");
    if (int rc = check_host_tables(h_sizes, h_bitrates, V, A, params)) return rc;
    if (int rc = check_mpc_shape(A, horizon)) return rc;
    if (mode != ABR_MPC_REF && mode != ABR_MPC_ROBUST) return fail(ABR_ERR_INVALID, "unknown MPC mode %d", mode);
    if (M < 0) return fail(ABR_ERR_RANGE, "M must be >= 0");
    if (n_history < 1) return fail(ABR_ERR_RANGE, "empty throughput history (ZeroDivisionError in mpc.py:90)");
    for (int j = 0; j < n_history; ++j)
        if (h_history[j] == 0.0) return fail(ABR_ERR_RANGE, "zero throughput sample (ZeroDivisionError in mpc.py:88)");
    if (chunk_idx < 0 || chunk_idx + horizon > V) return fail(ABR_ERR_RANGE, "chunk_idx + horizon exceeds the video (IndexError in mpc.py:125-128)");
    if (prev_q >= A) return fail(ABR_ERR_RANGE, "prev_q out of range");
    for (size_t i = 0; i < (size_t)M * horizon; ++i)
        if (h_sequences[i] < 0 || h_sequences[i] >= A) return fail(ABR_ERR_RANGE, "sequence entry %zu out of range", i);
    if (int rc = require_device()) return rc;
    std::vector<double> util;
    utility_table(h_bitrates, V, A, params, util);
    const size_t m = (size_t)(M > 0 ? M : 1);
    double* dd = nullptr;
    int32_t* di = nullptr;
    CUDA_TRY(cudaMalloc(&dd, sizeof(double) * (2 * (size_t)V * A + n_history + m)));
    if (cudaMalloc(&di, sizeof(int32_t) * m * horizon) != cudaSuccess) { cudaFree(dd); return fail(ABR_ERR_CUDA, "cudaMalloc failed"); }
    struct Free { double* a; int32_t* b; ~Free() { cudaFree(a); cudaFree(b); } } fr{dd, di};
    double* d_sizes = dd; double* d_util = d_sizes + (size_t)V * A; double* d_hist = d_util + (size_t)V * A;
    double* d_scores = d_hist + n_history;
    cudaStream_t st = 0;
    CUDA_TRY(cudaMemcpyAsync(d_sizes, h_sizes, sizeof(double) * V * A, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(d_util, util.data(), sizeof(double) * V * A, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(d_hist, h_history, sizeof(double) * n_history, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(di, h_sequences, sizeof(int32_t) * (size_t)M * horizon, cudaMemcpyHostToDevice, st));
    CUDA_TRY(launch_mpc_score(d_sizes, d_util, V, A, *params, chunk_idx, prev_q, buffer, d_hist, n_history, horizon, mode,
                              max_err, di, M, d_scores, st));
    CUDA_TRY(cudaMemcpyAsync(h_scores, d_scores, sizeof(double) * M, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return ABR_OK;
}

int abr_fp64_probe(int kind, int iters, double* gops_per_s, float* ms, void* stream) {
    if (iters < 1) return fail(ABR_ERR_RANGE, "iters must be >= 1");
    cudaStream_t st = (cudaStream_t)stream;
    if (kind >= 10) {   // latency probes: kind 10 DADD, 11 DMUL, 12 DADD+sign-mask; result = cycles per dependent op
        double* d_s = nullptr;
        long long* d_c = nullptr;
        CUDA_TRY(cudaMalloc(&d_s, sizeof(double) * 32));
        CUDA_TRY(cudaMalloc(&d_c, sizeof(long long)));
        struct F { double* a; long long* b; ~F() { cudaFree(a); cudaFree(b); } } f{d_s, d_c};
        CUDA_TRY(launch_fp64_latency(kind - 10, iters, d_s, d_c, st));
        CUDA_TRY(launch_fp64_latency(kind - 10, iters, d_s, d_c, st));
        long long cyc = 0;
        CUDA_TRY(cudaMemcpyAsync(&cyc, d_c, sizeof(cyc), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        if (gops_per_s) *gops_per_s = (double)cyc / ((double)iters * 64.0);
        if (ms) *ms = 0.f;
        return ABR_OK;
    }
    int dev = 0, sms = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    double* d_sink = nullptr;
    CUDA_TRY(cudaMalloc(&d_sink, sizeof(double) * (size_t)sms * 8 * 256));
    struct Free { double* p; ~Free() { cudaFree(p); } } fr{d_sink};
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0));
    CUDA_TRY(cudaEventCreate(&e1));
    int threads = 0;
    long long ops = 0;
    CUDA_TRY(launch_fp64_probe(kind, iters, d_sink, &threads, &ops, st));  // warm-up
    float best = 1e30f;
    for (int rep = 0; rep < 3; ++rep) {
        CUDA_TRY(cudaEventRecord(e0, st));
        CUDA_TRY(launch_fp64_probe(kind, iters, d_sink, &threads, &ops, st));
        CUDA_TRY(cudaEventRecord(e1, st));
        CUDA_TRY(cudaEventSynchronize(e1));
        float t = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&t, e0, e1));
        if (t < best) best = t;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (ms) *ms = best;
    if (gops_per_s) *gops_per_s = (double)threads * (double)ops / ((double)best * 1e-3) * 1e-9;
    return ABR_OK;
}

}  // extern "C"
