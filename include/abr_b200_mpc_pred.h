/* abr_b200_mpc_pred.h — MPC over caller-supplied throughput predictions (SPEC.md §5.6).
 *
 * abr_b200.h is the version-200 surface that existing bindings mirror entry for entry; this entry point is an
 * addition to it, declared in its own header so that those bindings stay complete as they are.  Same conventions as
 * abr_b200.h ("d_" device pointers, `stream` a cudaStream_t as void*, ABR_OK or an error code, abr_last_error()).
 */
#ifndef ABR_B200_MPC_PRED_H
#define ABR_B200_MPC_PRED_H
#include "abr_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* SPEC 5.6: the robust MPC decision (SPEC 5.2 objective, SPEC 5.5 branch and bound unless flags has
 * ABR_MPC_EXHAUSTIVE) for every session, over the caller's throughput predictions d_pred[s * horizon + i] for the
 * next h = min(horizon, V - chunk) chunks instead of the built-in predictor.  Only the first h entries of a row are
 * read; one that is not finite and > 0 is an input error for that session (action -1, counted once in the error
 * counter).  The history ring is not read and no state is written.  Rows are in environment order.
 * Checks, in this order: env not NULL (ABR_ERR_INVALID) and reset (ABR_ERR_STATE); an empty batch returns ABR_OK;
 * d_action, then d_pred not NULL, then flags 0 or ABR_MPC_EXHAUSTIVE (ABR_ERR_INVALID); horizon in [1, 8] and
 * A^horizon <= 2^31 - 1 (ABR_ERR_RANGE).  d_best_seq rows hold -1 past h. */
int abr_env_mpc_decide_pred(AbrEnv* env, int horizon, int flags, const double* d_pred /*[N][horizon]*/,
                            int32_t* d_action, double* d_best_j /*[N], nullable*/,
                            int32_t* d_best_seq /*[N][horizon], nullable*/, void* stream);

#ifdef __cplusplus
}
#endif
#endif
