/* abr_b200_dynamic.h — the DYNAMIC bitrate policy (SPEC.md §4.6): the rate rule while the buffer is low, BOLA once it
 * is high, with hysteresis between two buffer thresholds.
 *
 * abr_b200.h is the version-200 surface that existing bindings mirror entry for entry; these declarations are an
 * addition to it, declared in their own header so that those bindings stay complete as they are.  Same conventions
 * as abr_b200.h ("d_" device pointers, ABR_OK or an error code, abr_last_error()).
 *
 * ABR_POLICY_DYNAMIC is a policy id of the fused episode (abr_env_rollout_fused, _live, _f32, abr_env_run,
 * abr_env_run_host) and of abr_env_policy_decide.  It reads the throughput history, so it needs track_history = 1
 * (ABR_ERR_STATE otherwise), and BOLA's log table, so it needs every chunk size > 0 (ABR_ERR_INVALID otherwise),
 * checked in that order.
 */
#ifndef ABR_B200_DYNAMIC_H
#define ABR_B200_DYNAMIC_H
#include "abr_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

#define ABR_POLICY_DYNAMIC 5
/* abr_env_state_ptr field: the active rule of every session, uint8 [N] (0 = rate rule, 1 = BOLA), written only by
 * DYNAMIC decisions; zero when the environment is created with track_history = 1 (not allocated otherwise). */
#define ABR_F_DYN_MODE 24

/* The buffer thresholds of SPEC §4.6 in seconds: the rate rule hands over to BOLA when the pre-step buffer exceeds
 * switch_on_buffer [12 s], BOLA hands back when it no longer exceeds switch_off_buffer [6 s]. */
typedef struct AbrDynamicParams {
    double switch_on_buffer, switch_off_buffer;
} AbrDynamicParams;

void abr_dynamic_params_default(AbrDynamicParams* p);
/* Validates (finite 0 <= switch_off_buffer < switch_on_buffer; ABR_ERR_INVALID otherwise, before any device work and
 * before env is looked at) and installs them for the following calls.  abr_env_create installs the defaults.  The
 * rate and BOLA halves use the AbrPolicyParams of abr_env_set_policy_params. */
int abr_env_set_dynamic_params(AbrEnv* env, const AbrDynamicParams* params);

#ifdef __cplusplus
}
#endif
#endif
