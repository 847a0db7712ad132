/* abr_b200_obs.h — the windowed observation of the policy-in-the-loop step (SPEC.md §4.5).
 *
 * abr_b200.h is the version-200 surface that existing bindings mirror entry for entry; these entry points are an
 * addition to it, declared in their own header so that those bindings stay complete as they are.  Same conventions
 * as abr_b200.h ("d_" device pointers, `stream` a cudaStream_t as void*, ABR_OK or an error code, abr_last_error()).
 */
#ifndef ABR_B200_OBS_H
#define ABR_B200_OBS_H
#include "abr_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* The window length W in [1, 32] and the scales of the windowed observation obs[3 + 2W + A][N] (SPEC 4.5): row 0
 * the last chunk's utility * util_scale, row 1 the buffer * buffer_scale, row 2 the chunks left / V, rows 3 .. 3+W-1
 * the last W throughputs * throughput_scale and rows 3+W .. 3+2W-1 the last W download times * delay_scale (oldest
 * first, 0 before there are W), rows 3+2W .. the next chunk's sizes * size_scale. */
typedef struct AbrObsWindowSpec {
    int32_t window;
    double util_scale, buffer_scale, throughput_scale, delay_scale, size_scale;
} AbrObsWindowSpec;

/* SPEC 4.5: abr_env_step_policy (SPEC 4.1) with the windowed observation in place of the 4.1 one.  d_obs holds the
 * windows from one call to the next and is read and written in place: a step moves both windows up one entry and
 * appends its throughput and download time; a step that ends the video with auto_reset zeroes them; an inert step
 * (a done session, auto_reset = 0) leaves them.  Everything else is abr_env_step_policy bit for bit.
 * Checks, in this order: env not NULL (ABR_ERR_INVALID); reset, then not live mode (ABR_ERR_STATE); an empty batch
 * returns ABR_OK; d_logits, then spec, then d_obs not NULL (ABR_ERR_INVALID); spec->window in [1, 32]
 * (ABR_ERR_RANGE). */
int abr_env_step_policy_window(AbrEnv* env, const float* d_logits /*[N][A]*/, int sample, uint64_t seed,
                               const AbrObsWindowSpec* spec, float* d_obs /*[3 + 2W + A][N]*/,
                               int32_t* d_action_out /*[N], nullable*/, double* d_reward_sum /*[N], nullable*/,
                               double* d_delay, double* d_sleep, double* d_buffer, double* d_rebuf, double* d_reward,
                               uint8_t* d_end_of_video /*[N] each, nullable*/, void* stream);

/* SPEC 4.5: the windowed observation of the current state with both windows 0 (the first observation of an episode,
 * or a restart of the windows).  Writes nothing else.  Columns are in environment order.  Checks as
 * abr_env_step_policy_window, without d_logits. */
int abr_env_observe_window(AbrEnv* env, const AbrObsWindowSpec* spec, float* d_obs /*[3 + 2W + A][N]*/, void* stream);

#ifdef __cplusplus
}
#endif
#endif
