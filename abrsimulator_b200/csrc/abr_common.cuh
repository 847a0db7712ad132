// Internal definitions shared by the sm_100a kernels (abr_step.cu, abr_mpc.cu) and the C-ABI (abr_capi.cu).
// Arithmetic contract: SPEC.md.  All fp64 arithmetic goes through the _rn intrinsics below so that no
// FMA contraction or reassociation can happen regardless of compiler flags.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/abr_b200.h"

// Checked build (-DABR_CHECKED, `ABR_LIB_SUFFIX=_chk ABR_EXTRA_NVCC_FLAGS=-DABR_CHECKED`): every shared-memory and table
// access of the kernels is range-checked and a violation prints its location and traps, so the launch fails loudly.
// This is the repo's own memcheck: compute-sanitizer is not available on the GPU pool this was developed on.  The
// whole -m gpu suite is run against the checked library (profiles/README.md); the normal build compiles the checks away.
#ifdef ABR_CHECKED
#include <cstdio>
#define ABR_CHECK(cond, what)                                                                                          \
    do {                                                                                                               \
        if (!(cond)) {                                                                                                 \
            printf("ABR_CHECK failed: %s (%s:%d) block %d thread %d\n", what, __FILE__, __LINE__, (int)blockIdx.x,     \
                   (int)threadIdx.x);                                                                                  \
            __trap();                                                                                                  \
        }                                                                                                              \
    } while (0)
#else
#define ABR_CHECK(cond, what) do { } while (0)
#endif

namespace abr {

// Row stride (in doubles) of the cumulative-capacity table C[0..T] of SPEC §3.1: a multiple of four, so that every
// row starts 32-byte aligned (TMA bulk copies need 16; the global path reads aligned 256-bit quads), with at least
// seven entries of +inf padding behind C[T] (the global path's eight-entry window may start at C[T-1]).
__host__ __device__ __forceinline__ int cum_stride(int T_max) { return (T_max + 8 + 3) & ~3; }
// Bucket index of SPEC §3.1 (how the step finds the segment a download ends in; not part of the arithmetic contract):
// the trace period's data range [0, P) is cut into M = 2T equal cells, idx[b] = number of interior segment
// boundaries C[1..T-1] that lie in cells below b.  A position x in cell b then ends in a segment j with
// idx[b] <= j <= idx[b+1] — usually zero or one candidate boundary instead of a log2(T)-step search.
// 16-bit entries: traces longer than 65 535 segments get no index (M = 0) and are searched by bisection.
constexpr int kIdxMaxT = 65535;
__host__ __device__ __forceinline__ int idx_cells(int T) { return T <= kIdxMaxT ? 2 * T : 0; }
// Row stride (in 16-bit words) of the index table, M + 1 entries per row; a multiple of 8 (16-byte rows for TMA).
__host__ __device__ __forceinline__ int idx_stride(int T_max) { return T_max <= kIdxMaxT ? (2 * T_max + 2 + 7) & ~7 : 0; }
// Doubles a staged copy of a C row occupies in shared memory: the row plus two entries of slack (the step reads
// C[j0 .. j0+3] unconditionally and discards what lies past the candidates).
__host__ __device__ __forceinline__ int cum_smem_doubles(int T_max) { return cum_stride(T_max) + 2; }

// ---------------------------------------------------------------------------------------------
// exact fp64 helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double ddiv(double a, double b) { return __ddiv_rn(a, b); }

// Python `max(0, x)` (mpc.py:107): x if x > 0 else +0.  Done on the integer pipe (sign-bit mask) so
// that it does not take an FP64 issue slot: 1 shift + 2 logic ops instead of DSETP + 2 selects.
// Differs from the comparison form only for NaN inputs, which SPEC-valid inputs cannot produce.
__device__ __forceinline__ double max0(double x) {
    int hi = __double2hiint(x);
    int lo = __double2loint(x);
    int keep = ~(hi >> 31);
    return __hiloint2double(hi & keep, lo & keep);
}

// 1/d when d is a power of two in [2^-500, 2^500] (then x/d == x*(1/d) exactly for every finite x whose
// quotient is a normal number; the callers' operands are seconds, far from the fp64 range limits), else 0.
__device__ __forceinline__ double pow2_inverse(double d) {
    const int hi = __double2hiint(d), lo = __double2loint(d);
    const int e = (hi >> 20) & 0x7ff;
    if (lo != 0 || (hi & 0x800fffff) != 0 || e < 523 || e > 1523) return 0.0;
    return __hiloint2double((2046 - e) << 20, 0);
}

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 (SPEC §4); identical to oracle/abr_oracle.c:orc_philox4x32_10
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                               uint32_t k1) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(M0, c0), lo0 = M0 * c0;
        uint32_t hi1 = __umulhi(M1, c2), lo1 = M1 * c2;
        uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += W0; k1 += W1;
    }
    return make_uint4(c0, c1, c2, c3);
}

// ---------------------------------------------------------------------------------------------
// device-side view of an environment (passed by value to kernels)
// ---------------------------------------------------------------------------------------------
// What a step reads about its trace, packed so that it is one dependent 32-byte read after trace_id instead of
// four scattered ones (interval, period capacity C[T], length, search widths).
struct __align__(32) TraceMeta {
    double I, P;      // segment duration, capacity of one trace period C[T]
    double scale;     // M / P: cell of a data position x is (int)(x * scale), clamped to M - 1
    int32_t T, M;     // segments, index cells (0 = no index)
};

struct EnvView {
    // read-only tables
    const double* __restrict__ trace_bw;        // [n_traces][T_max]
    const double* __restrict__ trace_cum;       // [n_traces][cum_stride] C[0] = 0, C[j+1] = C[j] + (bw[j]*payload)*I (SPEC §3.1);
                                                // entries past C[T] are +inf
    const uint16_t* __restrict__ trace_idx;     // [n_traces][idx_stride] bucket index over C (see idx_cells)
    const TraceMeta* __restrict__ trace_meta;   // [n_traces] the per-trace scalars a step needs, one 32-byte record
    const int32_t* __restrict__ trace_len;      // [n_traces]
    const double* __restrict__ trace_interval;  // [n_traces]
    const double* __restrict__ sizes;           // [V][A]
    const double* __restrict__ util;            // [V][A]
    const double2* __restrict__ tab;            // [V][A] {size, utility}: one 16-byte read per step instead of two
    // SoA session state, capacity = cap
    int32_t* seg; int32_t* chunk; int32_t* last_q; int32_t* trace_id; int32_t* hist_len; int32_t* err_len;
    uint8_t* done; uint8_t* started;
    double* t_now; double* play_time;            // live mode (SPEC §7)
    int32_t* play_id; double* play_len;          // content chunk being played and how much of it has been played
    double* phi; double* pos; double* buffer; double* bw_hist; double* last_pred; double* err_ring; double* acc;
    const int32_t* perm;                        // session order (abr_env_set_order): caller's index of position i, or null
    unsigned long long* errors;                 // device counter of flagged sessions
    int n_traces, T_max, V, A, K, cap, n;       // n = active sessions
    int uniform_util;                           // every chunk has the same utility row (the usual case: one bitrate ladder)
    long long session_base;
    AbrParams p;
    // RATE / BOLA policies (SPEC §4.2, §4.3), derived on the host from AbrPolicyParams; last, so that the fields
    // above keep their kernel-parameter offsets
    struct Policy {
        const double* __restrict__ bola_v;      // [V][A] log(sizes[k][a] / sizes[k][0]); null when a size is not > 0
        double rb_safety, bola_Vp, bola_gp, bola_vmax;
        // DYNAMIC (SPEC §4.6): the per-session active rule (0 = RATE, 1 = BOLA; allocated with track_history = 1)
        // and the buffer thresholds that switch it; after the fields above for the same reason.  32 bytes with the
        // padding: the kernel parameters that follow an EnvView keep their 16-byte alignment, which the compiler uses
        // to load two of them at once (24 bytes turned such pairs into two loads in kernels that never read these).
        uint8_t* dyn_mode;
        double dyn_on, dyn_off;
        double pad_;
    } pol;
    // Catch-up speed control (SPEC §7.2): the speed of the chunk each live session is playing (allocated with
    // live = 1), the controller's parameters and whether it is installed.  Last and 64 bytes, for the reasons given
    // at Policy: the fields above keep their offsets and the parameters behind an EnvView their 16-byte alignment.
    struct SpeedControl {
        double* play_speed;
        double target_latency, max_drift, gain, dead_band, min_buffer;
        int32_t on;
        int32_t pad_[3];
    } spd;
    // Per-session policy parameters (SPEC §4.7, abr_env_set_session_policy_params): the environment's [kSessFields][cap]
    // table, row f of caller index c at f * cap + c (rows in the order of SessField), for the n sessions it was
    // installed for; used while `on`.  Last and 16 bytes, for the reasons given at Policy.
    struct SessionParams {
        const double* __restrict__ tab;
        int32_t n, on;
    } sp;
};

// Rows of EnvView::SessionParams::tab: the seven fields of AbrSessionPolicyParams in their order, then BOLA's (Vp, gp)
// derived from them as install_policy_params derives the environment-wide pair.
enum SessField { kSpBbaReservoir, kSpBbaCushion, kSpRbSafety, kSpBolaMin, kSpBolaTarget, kSpSwitchOn, kSpSwitchOff,
                 kSpBolaVp, kSpBolaGp, kSessFields };
// Bit OR-ed into the POLICY template argument of the episode and decision kernels: their forms with the per-session
// knobs of SPEC §4.7.
constexpr int kPolicySession = 16;

// launchers implemented in abr_step.cu / abr_mpc.cu (C++ linkage, internal)
cudaError_t launch_trace_table(const EnvView& v, double* d_cum, uint16_t* d_idx, int32_t* d_ok, TraceMeta* d_meta,
                               cudaStream_t st);
cudaError_t launch_reset(const EnvView& v, const int32_t* d_trace_id, const double* d_start_offset,
                         uint32_t* d_draw_counter, cudaStream_t st);
// Policy-in-the-loop step (abr_env_step_policy, SPEC §4.1): the action is drawn inside the step kernel from the
// caller's logits and the next observation is written by the same kernel.
struct StepPolicy {
    const float* __restrict__ logits = nullptr;    // [N][A] row-major scores of the caller's policy
    const uint32_t* __restrict__ draw = nullptr;   // device counter: index of this draw (Gumbel-max); null = greedy arg max
    uint32_t seed_lo = 0, seed_hi = 0;
    int32_t* __restrict__ action_out = nullptr;    // [N], nullable
    float* __restrict__ obs = nullptr;             // [4 + A][N] feature-major, nullable
    double s_buffer = 1.0, s_thr = 1.0, s_delay = 1.0, s_size = 1.0;   // observation scales
    double* __restrict__ reward_sum = nullptr;     // [N]: += reward, nullable
};
// SPEC §4.5 windowed observation (abr_env_step_policy_window, abr_env_observe_window): the StepPolicy fields, then
// window = W in [1, 32], which selects it (0 = the §4.1 observation), and its scales w_*; obs is then
// [3 + 2W + A][N] and carries the throughput and download-time windows from one call to the next.  A type of its own
// rather than fields appended to StepPolicy: a larger StepPolicy parameter changed the code of the live step kernels.
struct StepPolicyWindow : StepPolicy {
    int32_t window = 0;
    double w_util = 1.0, w_buffer = 1.0, w_thr = 1.0, w_delay = 1.0, w_size = 1.0;
};
// Per-step outputs of both step launchers: element ix of each array ([N] for a step, [steps][N] for an episode,
// next_sizes [N][A]); every pointer is nullable.  OT: double, or float for the fp32-output mode (the arithmetic stays
// fp64, an output is rounded once on the store).
template <typename OT>
struct StepOutputs {
    OT* __restrict__ delay = nullptr; OT* __restrict__ sleep = nullptr; OT* __restrict__ buffer = nullptr;
    OT* __restrict__ rebuf = nullptr; OT* __restrict__ reward = nullptr; uint8_t* __restrict__ eov = nullptr;
    int32_t* __restrict__ actions = nullptr;      // episode only: the action of every step
    OT* __restrict__ latency = nullptr;           // live mode (SPEC §7); the per-step kernel writes 0 outside it
    OT* __restrict__ thr = nullptr;               // per-step kernel only
    OT* __restrict__ next_sizes = nullptr;        // per-step kernel only
    // the five f64 outputs and end_of_video, which the FAST kernels store without null checks
    bool has_core() const { return delay && sleep && buffer && rebuf && reward && eov; }
    // no output at all: the NOOUT episode kernels
    bool none() const {
        return !delay && !sleep && !buffer && !rebuf && !reward && !eov && !actions && !latency && !thr && !next_sizes;
    }
};
cudaError_t launch_step_policy(const EnvView& v, const StepPolicyWindow& pol, const StepOutputs<double>& o,
                               uint32_t* d_draw_counter, cudaStream_t st);
// abr_env_observe_window (SPEC §4.5): the windowed observation of the state, both windows 0; pol.window and pol.obs set
cudaError_t launch_observe_window(const EnvView& v, const StepPolicyWindow& pol, cudaStream_t st);
// d_speed (live mode): the playback speed of content chunk k of session i is d_speed[k * N + i]; nullable = 1.0.
// With v.spd.on (live mode only) the catch-up controller of SPEC §7.2 decides the speeds instead; d_speed is null then.
template <typename OT>
cudaError_t launch_step(const EnvView& v, const int32_t* d_action, const double* d_speed, const StepOutputs<OT>& o,
                        cudaStream_t st, const StepPolicyWindow* policy = nullptr);
// Fused reset + episode + session cost (abr_env_run_host): with in_trace_id the episode kernel resets every session
// itself (SPEC §2) and out_cost receives Simulator.calculate_qoe per session; the pointers may alias pinned host memory.
// Scratch of the statistics reduction (SPEC §6): one sum per group of block partials, and the counters of finished
// blocks / groups (counters[0]: groups, counters[1 + g]: blocks of group g; zero between launches).
struct StatsScratch { double* group_partials = nullptr; unsigned int* counters = nullptr; };
// out_stats (with scratch): the statistics vector of SPEC §6 is written by the episode kernel itself (its last block).
struct RolloutFused {
    const int32_t* in_trace_id = nullptr; const double* in_offset = nullptr; double* out_cost = nullptr;
    double* out_stats = nullptr; StatsScratch scratch;
};
// step_base: episode steps since the last reset (the random policy's counter, SPEC §4)
template <typename OT>
cudaError_t launch_rollout(const EnvView& v, int policy, uint64_t seed, int steps, uint32_t step_base,
                           const int32_t* d_actions_in, const double* d_speed, const StepOutputs<OT>& o,
                           double* d_block_partials, const RolloutFused& f, cudaStream_t st);
// abr_env_policy_decide: the action of policy BBA / RATE / BOLA / DYNAMIC for every session from the SoA state
// (DYNAMIC also writes the session's active rule)
cudaError_t launch_policy_decide(const EnvView& v, int policy, int32_t* d_action, cudaStream_t st);
// abr_env_set_session_policy_params (SPEC §4.7): src[f] is the caller's [n] array of field f, or null for the
// environment-wide value env_wide[f].  With d_first: validation only, which sets *d_first to the smallest
// 8 * session + field that fails its check (all ones when none does) and writes nothing else.  Without: writes rows
// 0..6 of the [kSessFields][cap] table d_tab and derives rows 7 and 8.
struct SessionParamsSrc { const double* src[7]; double env_wide[7]; double bola_vmax; };
cudaError_t launch_session_params(const SessionParamsSrc& a, int n, int cap, double* d_tab,
                                  unsigned long long* d_first, cudaStream_t st);
// abr_env_lookahead_decide (SPEC §4.4): the clairvoyant best sequence over the next min(H, V - chunk) chunks against
// every session's own trace, H in [1, 8]; d_best_value [N] and d_best_seq [N][H] nullable.  Writes nothing else but
// the error counter.
cudaError_t launch_lookahead(const EnvView& v, int H, int32_t* d_action, double* d_best_value, int32_t* d_best_seq,
                             cudaStream_t st);
// abr_env_run_shared (SPEC §9): n_links links of G players, session l*G + p is player p of link l (v.n = n_links*G).
// policy: the built-in policy of player slot p in bits 4p .. 4p+3 (a packed value: the kernel selects by lane).  Writes the trajectory, request_time and the per-link outputs where
// non-null, the accumulators, qoe_cost (nullable) and the state of every player.
struct SharedRun {
    const int32_t* link_trace_id; const double* link_offset; const double* join_delay; const int32_t* actions_in;
    int n_links, G, steps;
    uint32_t seed_lo, seed_hi;
    uint32_t policy[4];
    StepOutputs<double> traj;   // [steps][N]: delay, sleep, buffer, rebuf, reward, eov, actions
    double* request_time;       // [steps][N]
    double *link_time, *link_capacity, *link_delivered, *qoe_cost;
};
cudaError_t launch_shared(const EnvView& v, const SharedRun& r, cudaStream_t st);
cudaError_t launch_stats(const EnvView& v, double* d_partials, int n_partials, bool have_partials, double* d_out,
                         const StatsScratch& scratch,
                         cudaStream_t st);
int stats_num_partials(int n);
int stats_num_groups(int n_partials);
void sort_shape(int n, int n_traces, int* S, int* n_blocks);
cudaError_t launch_gather(const int32_t* d_trace_id, const double* d_off, const int32_t* d_perm, int n,
                          int32_t* d_tid_sorted, double* d_off_sorted, cudaStream_t st);
cudaError_t launch_sort_gather(const int32_t* d_trace_id, const double* d_off, int n, int n_traces, int S, int n_blocks,
                               int32_t* d_hist, void* d_scan_tmp, size_t scan_tmp_bytes, int32_t* d_perm,
                               int32_t* d_tid_sorted, double* d_off_sorted, cudaStream_t st);
size_t sort_scan_tmp_bytes(int total);
cudaError_t launch_sort_by_trace(const int32_t* d_trace_id, int n, int n_traces, int32_t* d_perm, void* d_tmp,
                                 size_t* tmp_bytes, cudaStream_t st);
cudaError_t launch_qoe_cost(const EnvView& v, double* d_out, cudaStream_t st);
int rollout_num_blocks(int n);

struct MpcArgs {
    const double* sizes; const double* util; int V, A;
    AbrParams p;
    int N;
    const int32_t* chunk_idx; const int32_t* prev_q; const double* buffer; const uint8_t* done;  // done nullable
    const double* bw_hist; const int32_t* hist_len; int K;
    long long hist_session_stride, hist_slot_stride;       // element (s, slot) at s*session_stride + slot*slot_stride
    double* last_pred; double* err_ring; int32_t* err_len; // nullable; err ring uses the same strides
    int H, mode, flags;
    int32_t* action; double* best_j; int32_t* best_seq; double* preds;
    unsigned long long* error_count64; int32_t* error_count32; // either may be null
    // start-up phase (SPEC §5.3): sessions with startup[s] != 0 also choose a start-up delay on the grid jt * ts_step
    const uint8_t* startup = nullptr; int n_ts = 1; double ts_step = 0.0; double* startup_delay = nullptr;
    // caller-supplied predictions (SPEC §5.6): [N][H], p_i of session s at s*H + i; non-null selects the EXT kernels,
    // which read neither the history ring nor the robust state.  Last, so that every other field keeps its offset.
    const double* pred = nullptr;
};
cudaError_t launch_mpc(const MpcArgs& a, cudaStream_t st);
// MPC over throughput scenarios (SPEC §5.7): pred [N][K][H], weight [N][K] (nullable, MEAN only)
struct MpcScenArgs {
    const double* sizes; const double* util; int V, A;
    AbrParams p;
    int N;
    const int32_t* chunk_idx; const int32_t* prev_q; const double* buffer; const uint8_t* done;  // done nullable
    int H, K, objective, flags;
    const double* pred; const double* weight;
    int32_t* action; double* best_j; int32_t* best_seq;   // best_j, best_seq nullable
    unsigned long long* error_count64;
};
cudaError_t launch_mpc_scen(const MpcScenArgs& a, cudaStream_t st);
cudaError_t launch_mpc_score(const double* d_sizes, const double* d_util, int V, int A, const AbrParams& p, int k,
                             int prev_q, double buffer, const double* d_hist, int n, int H, int mode, double max_err,
                             const int32_t* d_seqs, int M, double* d_scores, cudaStream_t st);
cudaError_t launch_fp64_probe(int kind, int iters, double* d_sink, int* threads_total, long long* ops_per_thread,
                              cudaStream_t st);

cudaError_t launch_fp64_latency(int kind, int iters, double* d_sink, long long* d_cycles, cudaStream_t st);

void count_launch(int n = 1);

}  // namespace abr
