/* abr_b200_session_params.h — per-session policy parameters (SPEC.md §4.7): every session of a batch runs the built-in
 * policies BBA, RATE, BOLA and DYNAMIC with knobs of its own, e.g. a parameter sweep of G points in one launch.
 *
 * abr_b200.h is the version-200 surface that existing bindings mirror entry for entry; these declarations are an
 * addition to it, declared in their own header so that those bindings stay complete as they are.  Same conventions
 * as abr_b200.h ("d_" device pointers, ABR_OK or an error code, abr_last_error()).
 *
 * While parameters are installed, the BBA, RATE, BOLA and DYNAMIC decisions of abr_env_rollout_fused, _live, _f32,
 * abr_env_run, abr_env_run_host and abr_env_policy_decide use session s's values, s being the caller's index of the
 * session (its entry of the installed session order, or its position without one), in VoD, in live mode and with the
 * speed controller.  Those calls fail with ABR_ERR_STATE, after their other checks and before any device work, when
 * their session count (the active batch's; abr_env_run / _host: the call's n_sessions) is not the installed one.
 * ABR_POLICY_FIXED and _RANDOM ignore the parameters.  abr_env_set_policy_params and abr_env_set_dynamic_params fail
 * with ABR_ERR_STATE while parameters are installed (after their own checks).  With nothing installed every call
 * behaves as it does without this header.
 *
 * Storage: the environment owns one [capacity] array per field, plus BOLA's derived (Vp, gp), allocated at the first
 * installation.  The arrays never move; a later installation overwrites them in place.  A CUDA graph captured while
 * parameters are installed therefore replays with the values installed at replay time.
 */
#ifndef ABR_B200_SESSION_PARAMS_H
#define ABR_B200_SESSION_PARAMS_H
#include "abr_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Device pointers to [n_sessions] float64 arrays in caller order; NULL = the environment-wide value current at the
 * installation (bba_* from AbrParams, rb_safety and bola_* from abr_env_set_policy_params, switch_* from
 * abr_env_set_dynamic_params). */
typedef struct AbrSessionPolicyParams {
    const double *d_bba_reservoir, *d_bba_cushion, *d_rb_safety, *d_bola_min_buffer, *d_bola_target_buffer,
                 *d_switch_on_buffer, *d_switch_off_buffer;
} AbrSessionPolicyParams;

/* A non-NULL params installs the parameters of n_sessions sessions for the following calls; NULL removes them, which
 * restores the environment-wide behaviour bit for bit.  Checked in this order: NULL env (ABR_ERR_INVALID, without a
 * device); NULL params (removal, ABR_OK); n_sessions outside [1, capacity] (ABR_ERR_RANGE); then, on the device, per
 * session with the absent fields filled in: bba_reservoir finite, bba_cushion finite and > 0, rb_safety finite and
 * > 0, 0 < bola_min_buffer < bola_target_buffer (both finite), 0 <= switch_off_buffer < switch_on_buffer (both
 * finite).  A failure there is ABR_ERR_INVALID, naming the smallest failing session and its first failing field in
 * the order of AbrSessionPolicyParams.  The validation writes nothing and synchronises the stream: a failed call
 * leaves the previous installation exactly as it was. */
int abr_env_set_session_policy_params(AbrEnv* env, const AbrSessionPolicyParams* params, int n_sessions, void* stream);
/* The installed values (absent fields filled in) into d_out [7][n_sessions], rows in the order of
 * AbrSessionPolicyParams, caller order.  NULL env or d_out: ABR_ERR_INVALID; nothing installed: ABR_ERR_STATE;
 * n_sessions not the installed count: ABR_ERR_RANGE. */
int abr_env_get_session_policy_params(AbrEnv* env, double* d_out, int n_sessions, void* stream);

#ifdef __cplusplus
}
#endif
#endif
