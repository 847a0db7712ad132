/* abr_b200_lookahead.h — the clairvoyant lookahead of libabr_b200.so (SPEC.md §4.4).
 *
 * abr_b200.h is the version-200 surface that existing bindings mirror entry for entry; this entry point is an
 * addition to it, declared in its own header so that those bindings stay complete as they are.  Same conventions as
 * abr_b200.h ("d_" device pointers, `stream` a cudaStream_t as void*, ABR_OK or an error code, abr_last_error()).
 */
#ifndef ABR_B200_LOOKAHEAD_H
#define ABR_B200_LOOKAHEAD_H
#include "abr_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* SPEC 4.4: for every session, the first action of the bitrate sequence over the next min(H, V - chunk) chunks that
 * maximises the sum of the environment's own rewards against the session's actual future trace.  State unchanged.
 * An upper reference that sees the future, not a controller.  Checks, in this order: the env has been reset; not live
 * mode (ABR_ERR_STATE); an empty batch returns ABR_OK; d_action not NULL (ABR_ERR_INVALID); horizon in [1, 8] with
 * A^horizon <= 2^20 (ABR_ERR_RANGE).  d_best_seq rows hold -1 past min(H, V - chunk). */
int abr_env_lookahead_decide(AbrEnv* env, int horizon, int32_t* d_action, double* d_best_value /*[N], nullable*/,
                             int32_t* d_best_seq /*[N][horizon], nullable*/, void* stream);

#ifdef __cplusplus
}
#endif
#endif
