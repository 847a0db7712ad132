/* abr_b200_speed.h — catch-up speed control of live mode (SPEC.md §7.2): the playback speed of every content chunk is
 * decided when the chunk starts to play, from the session's latency and buffer at that instant.
 *
 * abr_b200.h is the version-200 surface that existing bindings mirror entry for entry; these declarations are an
 * addition to it, declared in their own header so that those bindings stay complete as they are.  Same conventions
 * as abr_b200.h ("d_" device pointers, ABR_OK or an error code, abr_last_error()).
 *
 * While a controller is installed, every live call plays with it in place of the [V][N] speed table: abr_env_step,
 * abr_env_step_live, abr_env_step_f32, abr_env_rollout_fused, _live, _f32, abr_env_run and abr_env_run_host.  Those
 * calls then reject a non-NULL d_speed with ABR_ERR_INVALID (a speed table and the speed controller are exclusive),
 * right after the reset check and before any device work.  With no controller installed every call behaves as it
 * does without this header.
 */
#ifndef ABR_B200_SPEED_H
#define ABR_B200_SPEED_H
#include "abr_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* abr_env_state_ptr field: the speed of the chunk each session is playing, float64 [N], written only by the
 * controller's decisions; zero when the environment is created with live = 1 (not allocated otherwise:
 * ABR_ERR_STATE). */
#define ABR_F_PLAY_SPEED 25

/* SPEC §7.2, with the latency error e = (wall clock - content played) - target_latency at the instant chunk k starts to
 * play and its buffer b:
 *     v = 1                                          if |e| <= dead_band
 *     v = 1 + max_drift * y / (1 + |y|), y = gain*e  otherwise
 *     v = 1                                          if v > 1 and b < min_buffer (never speed up into a stall)
 * Defaults (abr_speed_params_default): target_latency 12 s, max_drift 0.5, gain 2.5 /s, dead_band 0.02 s,
 * min_buffer 6 s. */
typedef struct AbrSpeedParams {
    double target_latency, max_drift, gain, dead_band, min_buffer;
} AbrSpeedParams;

void abr_speed_params_default(AbrSpeedParams* p);
/* A non-NULL params installs the controller for the following calls, NULL removes it.  Checked in this order before
 * any device work: params not finite or outside target_latency >= 0, 0 < max_drift < 1, gain > 0, dead_band >= 0,
 * min_buffer >= 0 (ABR_ERR_INVALID, also without a device); NULL env (ABR_ERR_INVALID); live = 0 (ABR_ERR_STATE). */
int abr_env_set_speed_control(AbrEnv* env, const AbrSpeedParams* params);

#ifdef __cplusplus
}
#endif
#endif
