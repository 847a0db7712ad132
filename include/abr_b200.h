/* abr_b200.h — C-ABI of the B200-native batched ABR environment and MPC controller.
 *
 * This is the drop-in boundary for the hot path of Elliotshui/ABRSimulator:
 * the per-session environment loop (Simulator.py:93-210) and the MPC bitrate
 * decision (mpc.py:69-186).  The reference is pure Python and has no FFI; the
 * entry points below are what a binding for that path would call (ctypes stub in
 * INTEGRATION.md).  Semantics of every call are fixed by SPEC.md.
 *
 * Conventions
 *  - plain pointers and sizes only; "d_" = device pointer on the current CUDA
 *    device, "h_" = host pointer.  The caller owns every buffer it passes; the
 *    library owns only the opaque AbrEnv (device copies of the tables + SoA
 *    session state).
 *  - `stream` is a cudaStream_t passed as void* (NULL = default stream).  Calls
 *    taking device pointers are asynchronous on that stream and never synchronise;
 *    calls with a "_host" suffix copy in/out and synchronise the stream before returning.
 *  - return value: ABR_OK (0) or an error code; abr_last_error() returns a
 *    thread-local message.  There is no CPU fallback: without a CUDA device every
 *    compute entry point fails with ABR_ERR_CUDA.
 *  - one AbrEnv per GPU/process; an AbrEnv is not thread-safe.
 */
#ifndef ABR_B200_H
#define ABR_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ABR_VERSION 200

enum { ABR_OK = 0, ABR_ERR_INVALID = 1, ABR_ERR_CUDA = 2, ABR_ERR_RANGE = 3, ABR_ERR_STATE = 4 };

/* built-in policies of the fused episode (SPEC §4): RATE is the rate-based rule (§4.2, needs track_history = 1),
 * BOLA the Lyapunov buffer rule (§4.3, needs every chunk size > 0) */
enum { ABR_POLICY_FIXED = 0, ABR_POLICY_RANDOM = 1, ABR_POLICY_BBA = 2, ABR_POLICY_RATE = 3, ABR_POLICY_BOLA = 4 };
/* MPC modes (SPEC §5): 0 = reference-exact mpc.py, 1 = robust MPC */
enum { ABR_MPC_REF = 0, ABR_MPC_ROBUST = 1 };
/* abr_mpc_decide flags */
enum { ABR_MPC_PRED_SES = 4,        /* mode 0: predictor "expsmoothing" (mpc.py:72-79) instead of "harmonic": the flat forecast of simple
                                      exponential smoothing, alpha = 0.5, least-squares initial level (SPEC 5.4) */
       ABR_MPC_TRUNCATE = 1,        /* mode 0: k+H > V truncates the horizon instead of flagging IndexError (mpc.py:125-128, D13) */
       ABR_MPC_EMPTY_DEFAULT = 2,   /* mode 0: empty history returns default_quality instead of flagging ZeroDivisionError (mpc.py:90, D14) */
       ABR_MPC_EXHAUSTIVE = 8 };    /* mode 1: evaluate every one of the A^H sequences, as scipy.optimize.brute does (mpc.py:171-179),
                                       instead of skipping the partial sequences whose bound already loses (branch and bound:
                                       the decision, its objective value and the first-minimum tie-break are the same) */
/* abr_env_mpc_decide takes the mode alone: OR this bit into it for the exhaustive enumeration */
#define ABR_MPC_MODE_EXHAUSTIVE 0x100

/* rows of the accumulator table / entries of the statistics vector (SPEC §6) */
enum { ABR_ACC_REWARD = 0, ABR_ACC_REBUF = 1, ABR_ACC_UTILITY = 2, ABR_ACC_SMOOTH = 3, ABR_ACC_SLEEP = 4,
       ABR_ACC_DELAY = 5, ABR_ACC_STEPS = 6, ABR_ACC_EPISODES = 7, ABR_ACC_STARTUP = 8,
       ABR_ACC_LATENCY = 9, /* live mode: integral of the latency over the time spent playing (SPEC §7) */
       ABR_ACC_PLAY = 10,   /* live mode: content played */
       ABR_NUM_ACC = 11, ABR_NUM_STATS = 11 };

/* session-state fields exposed by abr_env_state_ptr (SPEC §1).  All arrays have max_sessions elements except
 * BW_HIST / ERR_RING ([hist_k][max_sessions]) and ACC ([ABR_NUM_ACC][max_sessions]). */
enum { ABR_F_SEG = 0, ABR_F_CHUNK = 1, ABR_F_LAST_Q = 2, ABR_F_TRACE_ID = 3, ABR_F_HIST_LEN = 4, ABR_F_DONE = 5,
       ABR_F_ERR_LEN = 6, ABR_F_PHASE = 10, ABR_F_POS = 18, ABR_F_BUFFER = 11, ABR_F_BW_HIST = 12, ABR_F_LAST_PRED = 13,
       ABR_F_ERR_RING = 14, ABR_F_ACC = 15, ABR_F_T_NOW = 16, ABR_F_PLAY_TIME = 17, ABR_F_STARTED = 7,
       ABR_F_PLAY_ID = 8, ABR_F_PLAY_LEN = 19, ABR_F_SIZES = 20, ABR_F_UTILITY = 21, ABR_F_TRACE_BW = 22,
       ABR_F_ORDER = 23 /* the installed session order, int32 [N] (abr_env_set_order / abr_env_reset_sorted) */ };

/* Replaces the attribute bags MPD / QOEMetric (Simulator.py:11-24, mpc_test.py:18-29) plus the
 * north-star constants (SPEC §1). */
typedef struct AbrParams {
    double chunk_length;    /* MPD.chunk_length, Simulator.py:13 */
    double max_buffer;      /* MPD.max_buffer, Simulator.py:14 */
    double rtt;             /* added to every download delay */
    double payload;         /* packet-payload fraction applied to the trace bandwidth */
    double sleep_quantum;   /* sleep granularity while buffer > max_buffer */
    double rebuf_penalty;   /* QOEMetric.rebuffer_weight, Simulator.py:21 */
    double smooth_penalty;  /* QOEMetric.variance_weight, Simulator.py:22 */
    double utility_scale;   /* utility_mode 0: U = bitrate * utility_scale (1.0 = mpc.py:95-97 identity) */
    double bba_reservoir, bba_cushion;
    double start_up_length; /* live mode: buffer that ends the start-up phase, MPD.start_up_length, Simulator.py:12,201-202 */
    double startup_penalty; /* QOEMetric.startup_weight, Simulator.py:23 (session cost only) */
    double latency_penalty; /* QOEMetric.latency_weight, Simulator.py:24 (per-step reward and session cost) */
    double latency_tick;    /* live mode: the reference's tick (Simulator.py:133): its average_latency is the latency integral
                               over the playing time divided by (tick * content played), Simulator.py:179-180 */
    int32_t utility_mode;   /* 0 linear, 1 log(bitrate / top bitrate) (mpc.py:99-102) */
    int32_t default_quality;
    int32_t auto_reset;     /* 1: a session restarts at chunk 0 after its last chunk */
    int32_t hist_k;         /* capacity of the throughput-history ring (robust-MPC window) */
    int32_t track_history;  /* 1: abr_env_step / rollout push size/delay into the ring */
    int32_t track_acc;      /* 1: abr_env_step adds into the per-session accumulators */
    int32_t live;           /* 1: live-streaming semantics of SPEC §7 */
    int32_t smooth_prev_ladder; /* smoothness term |U[k][q_k] - U[k'][q_{k-1}]|: 0: k' = k (the current chunk's ladder,
                               mpc.py:148-149); 1: k' = k-1 (each chunk's own ladder, Simulator.calculate_qoe, Simulator.py:81-82) */
} AbrParams;

typedef struct AbrEnv AbrEnv;

/* ---- library ---- */
int abr_version(void);
const char* abr_last_error(void);
/* number of kernels this library has launched in this process (bench.py "gpu_launches") */
long long abr_launch_count(void);
int abr_device_info(int* sm_count, int* cc_major, int* cc_minor, long long* total_mem_bytes);
void abr_params_default(AbrParams* p);

/* ---- environment (replaces Simulator.set_network_info / set_mpd / set_qoe_metric + run,
 *      Simulator.py:54-77,93-210).  Table pointers are HOST pointers; they are validated
 *      (bandwidth finite and > 0, sizes finite and >= 0) and copied to the device. ---- */
int abr_env_create(const double* h_trace_bw /*[n_traces][T_max]*/, const int32_t* h_trace_len /*[n_traces]*/,
                   const double* h_trace_interval /*[n_traces]*/, int n_traces, int T_max,
                   const double* h_sizes /*[V][A]*/, const double* h_bitrates /*[V][A]*/, int V, int A,
                   const AbrParams* params, int max_sessions, AbrEnv** out);
void abr_env_destroy(AbrEnv* env);
int abr_env_num_sessions(const AbrEnv* env);
/* Session order.  Sessions are independent (the reference's Simulator holds exactly one, Simulator.py:93-131), so the
 * order in which an environment keeps them is free; kept sorted by trace, every thread block of the step kernels follows
 * one trace and stages it in shared memory whatever order the caller's sessions come in.
 * abr_sort_by_trace: d_perm[p] = caller's index of the session at environment position p (stable sort by trace id,
 * an invalid id (< 0 or >= n_traces) sorting as trace 0, deterministic; run once per session->trace assignment;
 * SPEC §8).
 * abr_env_set_order: installs (copies) such an order; NULL removes it.  Every per-session array the caller passes or
 * receives afterwards (trace ids, start offsets, actions, speeds, outputs, state views) is in ENVIRONMENT order, i.e.
 * element p belongs to the caller's session d_perm[p]; the only thing the library does with the order is key the
 * random policy by session_base + d_perm[p], so that a reordered run draws exactly the actions of the original one. */
int abr_sort_by_trace(const int32_t* d_trace_id, int n_sessions, int n_traces, int32_t* d_perm, void* stream);
int abr_env_set_order(AbrEnv* env, const int32_t* d_perm /*nullable*/, int n_sessions, void* stream);
/* SPEC §2.  session_base = global index of local session 0 (sharded runs; keys the random policy). */
int abr_env_reset(AbrEnv* env, const int32_t* d_trace_id, const double* d_start_offset /*nullable*/, int n_sessions,
                  long long session_base, void* stream);
/* abr_sort_by_trace + abr_env_set_order + abr_env_reset in one call, for sessions given in the CALLER's order: a
 * counting sort by trace (stable: the same order as abr_sort_by_trace) that gathers the trace ids and start offsets
 * into that order on the way, then the reset.  The order is readable afterwards with abr_env_get_order. */
int abr_env_reset_sorted(AbrEnv* env, const int32_t* d_trace_id, const double* d_start_offset /*nullable*/,
                         int n_sessions, long long session_base, void* stream);
/* Copies the installed order (n_sessions entries) to d_perm; ABR_ERR_STATE without one. */
int abr_env_get_order(AbrEnv* env, int32_t* d_perm, int n_sessions, void* stream);
int abr_env_reset_host(AbrEnv* env, const int32_t* h_trace_id, const double* h_start_offset /*nullable*/,
                       int n_sessions, long long session_base, void* stream);
/* SPEC §3: one chunk step for every session.  Output pointers are nullable. */
int abr_env_step(AbrEnv* env, const int32_t* d_action, double* d_delay, double* d_sleep, double* d_buffer,
                 double* d_rebuf, double* d_reward, double* d_next_sizes /*[N][A]*/, uint8_t* d_end_of_video,
                 double* d_throughput, void* stream);
/* SPEC §4.1 — policy-in-the-loop step for RL harnesses (BASELINE.json configs[4]; the reference's controller protocol
 * get_next_bitrate(...), Simulator.py:155, answered by a batched policy network): d_logits[N][A] are the policy's
 * scores for every session; the step kernel itself picks the action — arg max (sample = 0), or a draw from
 * softmax(logits) by Gumbel-max with Philox noise keyed by (seed, global session index, draw counter) (sample = 1; the
 * environment's draw counter is advanced by every sampled call and zeroed by abr_env_reset) — steps the session, adds
 * the reward into d_reward_sum[N] and writes the next observation d_obs[4 + A][N] (fp32, feature-major):
 *   row 0 buffer * buffer_scale, row 1 throughput of the download (size / delay) * throughput_scale,
 *   row 2 delay * delay_scale, row 3 action / A, rows 4.. sizes of the next chunk * size_scale.
 * Everything but d_logits is nullable.  Not available in live mode. */
typedef struct AbrObsSpec { double buffer_scale, throughput_scale, delay_scale, size_scale; } AbrObsSpec;
int abr_env_step_policy(AbrEnv* env, const float* d_logits, int sample, uint64_t seed, const AbrObsSpec* spec,
                        float* d_obs, int32_t* d_action_out, double* d_reward_sum, double* d_delay, double* d_sleep,
                        double* d_buffer, double* d_rebuf, double* d_reward, uint8_t* d_end_of_video, void* stream);
/* SPEC §7 (live = 1): like abr_env_step with the playback speeds as a second action and the latency output; d_sleep
 * receives the idle time before the download.  d_speed is a [V][N] table (nullable = 1.0): d_speed[k][s] is the speed
 * at which session s plays content chunk k — the reference asks its speed controller once per PLAYED chunk
 * (speed_controller.get_next_speed(), Simulator.py:176-177), so playback during one download may run at several
 * speeds; a caller that decides step by step rewrites the rows of the chunks not yet played between two calls.
 * With live = 0 it behaves like abr_env_step and writes 0 latency. */
int abr_env_step_live(AbrEnv* env, const int32_t* d_action, const double* d_speed, double* d_delay, double* d_sleep,
                      double* d_buffer, double* d_rebuf, double* d_reward, double* d_latency,
                      double* d_next_sizes /*[N][A]*/, uint8_t* d_end_of_video, double* d_throughput, void* stream);
/* SPEC §3+§4: `steps` chunk steps in one launch, state in registers.  Trajectory outputs are
 * [steps][N] and nullable; per-session sums are added into the env accumulators (ABR_F_ACC). */
int abr_env_rollout_fused(AbrEnv* env, int policy, uint64_t seed, int steps, const int32_t* d_actions_in,
                          double* d_delay, double* d_sleep, double* d_buffer, double* d_rebuf, double* d_reward,
                          uint8_t* d_end_of_video, int32_t* d_actions_out, void* stream);
/* The same episode with the live-streaming outputs (SPEC §7, live = 1): d_speed is the [V][N] playback-speed table
 * of abr_env_step_live (nullable = 1.0), d_latency the per-step latency ([steps][N], nullable), d_sleep the idle time
 * before each download.  With live = 0 it is abr_env_rollout_fused and both extra pointers must be NULL;
 * abr_env_rollout_fused on a live environment plays every session at speed 1. */
int abr_env_rollout_fused_live(AbrEnv* env, int policy, uint64_t seed, int steps, const int32_t* d_actions_in,
                               const double* d_speed, double* d_delay, double* d_sleep, double* d_buffer,
                               double* d_rebuf, double* d_reward, double* d_latency, uint8_t* d_end_of_video,
                               int32_t* d_actions_out, void* stream);
/* One whole run per call, device-resident: abr_env_reset + abr_env_rollout_fused + abr_env_qoe_cost +
 * abr_stats_partial in ONE launch — the episode kernel resets every session itself (SPEC §2, same operations as
 * abr_env_reset), writes the per-session cost and reduces the statistics (SPEC §6; the block that finishes last writes
 * them), so the state makes no round trip through HBM in between.
 * This is Simulator.run() (Simulator.py:93-210) for a batch: d_qoe_cost[N] is what run() returns per session
 * (calculate_qoe, Simulator.py:83-86).  Trajectory outputs [steps][N], d_qoe_cost and d_stats are nullable. */
int abr_env_run(AbrEnv* env, int policy, uint64_t seed, int steps, const int32_t* d_trace_id,
                const double* d_start_offset /*nullable*/, int n_sessions, long long session_base,
                const int32_t* d_actions_in /*[steps][N], policy FIXED*/, double* d_delay, double* d_sleep,
                double* d_buffer, double* d_rebuf, double* d_reward, uint8_t* d_end_of_video, int32_t* d_actions_out,
                double* d_qoe_cost /*[N]*/, double* d_stats /*[ABR_NUM_STATS]*/, void* stream);
/* Optional fp32-output mode (BASELINE.json north star: "1e-5 for an optional fp32 mode").  State, tables and every
 * arithmetic operation stay fp64 (SPEC §3), so trajectories do not drift; each floating-point output is rounded once
 * to float on the store (relative error <= 2^-24 = 6e-8 of the fp64 value).  The trajectory of a fused episode
 * shrinks from 41 to 21 B per chunk-step.  Signatures otherwise as abr_env_step_live / abr_env_rollout_fused_live
 * (d_speed / d_latency NULL unless live = 1). */
int abr_env_step_f32(AbrEnv* env, const int32_t* d_action, const double* d_speed, float* d_delay, float* d_sleep,
                     float* d_buffer, float* d_rebuf, float* d_reward, float* d_latency,
                     float* d_next_sizes /*[N][A]*/, uint8_t* d_end_of_video, float* d_throughput, void* stream);
int abr_env_rollout_fused_f32(AbrEnv* env, int policy, uint64_t seed, int steps, const int32_t* d_actions_in,
                              const double* d_speed, float* d_delay, float* d_sleep, float* d_buffer, float* d_rebuf,
                              float* d_reward, float* d_latency, uint8_t* d_end_of_video, int32_t* d_actions_out,
                              void* stream);
/* Parameters of the RATE and BOLA policies (SPEC §4.2, §4.3), kept apart from AbrParams so that its layout stays put.
 * rb_safety: the budget is rb_safety * harmonic mean * chunk_length [1.0].  bola_min_buffer / bola_target_buffer: the
 * buffer below which BOLA picks the lowest quality and at which the highest quality's score reaches zero [10, 30 s];
 * the paper's (V, gamma*p) are V = min / gp and gp = v_max / (target / min - 1). */
typedef struct AbrPolicyParams { double rb_safety, bola_min_buffer, bola_target_buffer; } AbrPolicyParams;
void abr_policy_params_default(AbrPolicyParams* p);
/* Validates (rb_safety finite and > 0, 0 < bola_min_buffer < bola_target_buffer, both finite; ABR_ERR_INVALID
 * otherwise, before any device work) and installs them for the following calls.  abr_env_create installs the defaults. */
int abr_env_set_policy_params(AbrEnv* env, const AbrPolicyParams* params);
/* The action of a built-in state-dependent policy (ABR_POLICY_BBA, _RATE or _BOLA) for every session, from the
 * environment's own state: the per-step counterpart of the fused episode's policies, to be followed by abr_env_step,
 * abr_env_step_live or abr_env_step_f32.  d_action[N] receives them.  FIXED, RANDOM and unknown ids: ABR_ERR_INVALID. */
int abr_env_policy_decide(AbrEnv* env, int policy, int32_t* d_action, void* stream);
/* MPC decision for every session from the env's own state and history ring (SPEC §5);
 * never flags errors (implies ABR_MPC_TRUNCATE | ABR_MPC_EMPTY_DEFAULT). */
int abr_env_mpc_decide(AbrEnv* env, int horizon, int mode, int32_t* d_action, double* d_best_j /*nullable*/,
                       void* stream);
/* Per-session QoE cost of Simulator.calculate_qoe (Simulator.py:83-86) from the accumulators into d_out[N]:
 * rw*rebuffer + vw*smooth + sw*startup + lw*average_latency, average_latency = latency integral / (latency_tick * content
 * played) as the reference's running mean defines it (Simulator.py:179-180; SPEC 7). */
int abr_env_qoe_cost(AbrEnv* env, double* d_out, void* stream);
/* SPEC §6: reduce the accumulators of the first n sessions into d_out[ABR_NUM_STATS]. */
int abr_stats_partial(AbrEnv* env, double* d_out, void* stream);
int abr_env_state_ptr(AbrEnv* env, int field, void** d_ptr);
/* sessions flagged so far (walk guard hit, invalid action, MPC input error); synchronises the stream */
int abr_env_error_count(AbrEnv* env, long long* out, void* stream);

/* ---- host-buffer entry points: what Simulator.run() (Simulator.py:93-210) and
 *      MPCBitrateController.next_bitrate() (mpc.py:181-186) callers use.  They copy inputs
 *      host->device, run the kernels above and copy results device->host.
 *      abr_env_run_host is abr_env_run with host buffers.  Buffers in page-locked memory (cudaHostAlloc /
 *      cudaHostRegister, e.g. torch's pin_memory()) are not copied: the episode kernel reads h_trace_id /
 *      h_start_offset and writes h_qoe_cost / h_stats through their device aliases, over PCIe, while other
 *      thread blocks compute.  Pageable buffers go through staged cudaMemcpyAsync.  Synchronises the stream. ---- */
int abr_env_run_host(AbrEnv* env, int policy, uint64_t seed, int steps, const int32_t* h_trace_id,
                     const double* h_start_offset, int n_sessions, long long session_base,
                     const int32_t* h_actions_in /*[steps][N], policy FIXED*/,
                     double* h_acc /*[ABR_NUM_ACC][N], nullable*/, double* h_stats /*[ABR_NUM_STATS], nullable*/,
                     double* h_reward_traj /*[steps][N], nullable*/,
                     double* h_qoe_cost /*[N], nullable: calculate_qoe per session, Simulator.py:83-86*/, void* stream);

/* ---- standalone MPC (replaces MPCBitrateController.next_bitrate over a batch of players,
 *      mpc.py:164-186).  Tables are device pointers [V][A].  History is a per-session ring
 *      [N][K]: slot (hist_len-1) mod K is the newest sample; hist_len <= K is a plain
 *      oldest-first row.  d_last_pred/d_err_ring/d_err_len ([N],[N][K],[N]) hold the robust
 *      error state (mode 1; nullable = no discount).  On an input error the action is -1
 *      and *d_error_count is incremented.  Outputs other than d_action are nullable. ---- */
int abr_mpc_decide(const double* d_sizes, const double* d_utility, int V, int A, const AbrParams* params, int N,
                   const int32_t* d_chunk_idx, const int32_t* d_prev_q, const double* d_buffer,
                   const double* d_bw_hist, const int32_t* d_hist_len, int K, double* d_last_pred,
                   double* d_err_ring, int32_t* d_err_len, int horizon, int mode, int flags, int32_t* d_action,
                   double* d_best_j, int32_t* d_best_seq /*[N][H]*/, double* d_preds /*[N][H]*/,
                   int32_t* d_error_count, void* stream);
/* Start-up phase of the controller (f_st of the pseudo-code at mpc.py:7-18; the reference leaves its start-up delay
 * at 0, "TODO", mpc.py:141, and weighs it with startup_weight, mpc.py:160).  SPEC 5.3: sessions with d_startup[s] != 0
 * (NULL = all) choose, besides the bitrate sequence, a start-up delay T_s on the grid {0, ts_step, ..., (n_ts-1)*ts_step}:
 * T_s is credited to the initial buffer of the lookahead and charged params->startup_penalty * T_s; d_startup_delay[N]
 * receives the chosen T_s ("start playback after T_s seconds"), 0 for sessions outside the start-up phase. */
int abr_mpc_decide_startup(const double* d_sizes, const double* d_utility, int V, int A, const AbrParams* params, int N,
                           const int32_t* d_chunk_idx, const int32_t* d_prev_q, const double* d_buffer,
                           const double* d_bw_hist, const int32_t* d_hist_len, int K, double* d_last_pred,
                           double* d_err_ring, int32_t* d_err_len, int horizon, int mode, int flags,
                           const uint8_t* d_startup, int n_ts, double ts_step, int32_t* d_action,
                           double* d_startup_delay, double* d_best_j, int32_t* d_best_seq, double* d_preds,
                           int32_t* d_error_count, void* stream);
int abr_mpc_decide_startup_host(const double* h_sizes, const double* h_bitrates, int V, int A, const AbrParams* params,
                                int N, const int32_t* h_chunk_idx, const int32_t* h_prev_q, const double* h_buffer,
                                const double* h_bw_hist, const int32_t* h_hist_len, int K, double* h_last_pred,
                                double* h_err_ring, int32_t* h_err_len, int horizon, int mode, int flags,
                                const uint8_t* h_startup, int n_ts, double ts_step, int32_t* h_action,
                                double* h_startup_delay, double* h_best_j, int32_t* h_best_seq, double* h_preds,
                                int32_t* h_error_count);
/* Host-buffer decisions stage through one arena per host thread (grow-only): a call is one host->device copy, one
 * kernel launch and one device->host copy, without any allocation once the arena has its size. */
int abr_mpc_decide_host(const double* h_sizes, const double* h_bitrates, int V, int A, const AbrParams* params, int N,
                        const int32_t* h_chunk_idx, const int32_t* h_prev_q, const double* h_buffer,
                        const double* h_bw_hist, const int32_t* h_hist_len, int K, double* h_last_pred,
                        double* h_err_ring, int32_t* h_err_len, int horizon, int mode, int flags, int32_t* h_action,
                        double* h_best_j, int32_t* h_best_seq, double* h_preds, int32_t* h_error_count);

/* objective() of caller-given sequences for ONE decision state (replaces MPCBitrateController.objective,
 * mpc.py:120-162): scores[m] = J(sequences[m][0..H-1]).  h_history is oldest first.  mode 1 uses
 * c = harmonic_mean / (1 + max_err).  Requires chunk_idx + horizon <= V and a non-empty, non-zero history. */
int abr_mpc_score_host(const double* h_sizes, const double* h_bitrates, int V, int A, const AbrParams* params,
                       int chunk_idx, int prev_q, double buffer, const double* h_history, int n_history, int horizon,
                       int mode, double max_err, const int32_t* h_sequences /*[M][H]*/, int M, double* h_scores /*[M]*/);

/* ---- measurement helper: FP64 issue-rate probe used as the MPC kernel's roofline denominator.
 *      kind 0 = dependent DADD chains, 1 = DFMA chains, 2 = DADD + DSETP/select mix.
 *      Returns giga-ops/s (one op per thread-instruction; FMA counts 1).
 *      kind 10/11/12 = latency probes (one dependent DADD / DMUL / DADD+sign-mask chain in one warp): the value
 *      returned in *gops_per_s is then SM cycles per dependent operation. ---- */
int abr_fp64_probe(int kind, int iters, double* gops_per_s, float* ms, void* stream);

#ifdef __cplusplus
}
#endif
#endif
