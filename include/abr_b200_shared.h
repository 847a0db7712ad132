/* abr_b200_shared.h — shared bottleneck links (SPEC.md §9): G players share one trace's capacity equally while their
 * downloads overlap (processor sharing), simulated event by event, one link per warp, in one launch per batch of links.
 *
 * abr_b200.h is the version-200 surface that existing bindings mirror entry for entry; these declarations are an
 * addition to it, declared in their own header so that those bindings stay complete as they are.  Same conventions
 * as abr_b200.h ("d_" device pointers, "h_" host pointers, ABR_OK or an error code, abr_last_error()).
 *
 * Batch shape: n_links links of G = players_per_link players; player p of link l is session l*G + p, so the run
 * covers n_sessions = n_links*G sessions.  Link l plays trace d_link_trace_id[l] from d_link_offset[l] (NULL = 0);
 * every player starts with the session state of a reset (SPEC §2) and makes exactly `steps` downloads.
 *
 * Afterwards the environment holds the batch as after abr_env_run: abr_env_qoe_cost, abr_stats_partial and the state
 * fields work on the n_sessions players; each player's seg / phase / pos is its link's final position.
 */
#ifndef ABR_B200_SHARED_H
#define ABR_B200_SHARED_H
#include "abr_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Outputs of abr_env_run_shared; every pointer is nullable.  Per player, [steps][n_sessions] (element k*N + s is
 * download k of session s): the step outputs of abr_env_run and request_time, the link clock when the download was
 * requested.  Per link, [n_links]: link_time, the clock when the link's last player finished; link_capacity, the data
 * the trace offered from the start to link_time; link_delivered, the sum of the downloaded sizes. */
typedef struct AbrSharedOutputs {
    double *d_delay, *d_sleep, *d_buffer, *d_rebuf, *d_reward, *d_request_time;
    uint8_t* d_end_of_video;
    int32_t* d_actions;
    double *d_link_time, *d_link_capacity, *d_link_delivered;
} AbrSharedOutputs;

/* SPEC §9.  policy: the built-in policy of every player, or, with h_player_policy (host, [players_per_link]), slot p of
 * every link runs h_player_policy[p] and `policy` is ignored.  d_join_delay [n_sessions] (NULL = 0): the time from the
 * link's start to each player's first request.  RANDOM draws are keyed by session_base + session and the download
 * index; FIXED reads d_actions_in [steps][n_sessions].  d_qoe_cost [n_sessions] and d_stats [ABR_NUM_STATS] are
 * nullable; d_stats equals abr_stats_partial afterwards.
 * Checked in this order, before any device work: NULL env or NULL d_link_trace_id with n_links > 0 (ABR_ERR_INVALID);
 * live mode, then an installed session order (ABR_ERR_STATE); players_per_link outside [1, 32], n_links < 0,
 * n_links*players_per_link above the capacity, steps < 0 (ABR_ERR_RANGE); then per player slot, the policy checks of
 * abr_env_run (an unknown policy and BOLA / DYNAMIC without positive sizes: ABR_ERR_INVALID; RATE / DYNAMIC without
 * track_history: ABR_ERR_STATE; FIXED without d_actions_in: ABR_ERR_INVALID); then the session count of installed
 * per-session policy parameters (ABR_ERR_STATE).  On the device, a negative or non-finite join delay counts the player
 * once in the error counter and the player joins at 0. */
int abr_env_run_shared(AbrEnv* env, int policy, const int32_t* h_player_policy, uint64_t seed, int steps,
                       int players_per_link, const int32_t* d_link_trace_id, const double* d_link_offset,
                       const double* d_join_delay, int n_links, long long session_base, const int32_t* d_actions_in,
                       const AbrSharedOutputs* out, double* d_qoe_cost, double* d_stats, void* stream);

#ifdef __cplusplus
}
#endif
#endif
