/* abr_b200_mpc_scen.h — MPC over caller-supplied throughput scenarios (SPEC.md §5.7).
 *
 * abr_b200.h is the version-200 surface that existing bindings mirror entry for entry; this entry point is an
 * addition to it, declared in its own header so that those bindings stay complete as they are.  Same conventions as
 * abr_b200.h ("d_" device pointers, `stream` a cudaStream_t as void*, ABR_OK or an error code, abr_last_error()).
 */
#ifndef ABR_B200_MPC_SCEN_H
#define ABR_B200_MPC_SCEN_H
#include "abr_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

#define ABR_MPC_SCEN_MEAN  0   /* the best weighted mean of the scenarios' objective values */
#define ABR_MPC_SCEN_WORST 1   /* the best worst case over the scenarios */
#define ABR_MPC_SCEN_MAX   16  /* most scenarios per session */

/* SPEC 5.7: for every session, the bitrate sequence over the next h = min(horizon, V - chunk) chunks whose SPEC 5.2
 * objective values under the n_scen throughput scenarios d_pred[(s * n_scen + k) * horizon + i] aggregate best:
 * weighted mean (weights d_weight[s * n_scen + k], or 1 / n_scen each when NULL) or worst case.  SPEC 5.5 branch and
 * bound unless flags has ABR_MPC_EXHAUSTIVE.  Only the first h entries of a scenario are read; one that is not finite
 * and > 0, or a weight that is not finite and >= 0, or all weights 0, is an input error for that session (action -1,
 * counted once in the error counter).  The history ring is not read and no state is written.  Rows are in
 * environment order.
 * Checks, in this order: env not NULL (ABR_ERR_INVALID) and reset (ABR_ERR_STATE); an empty batch returns ABR_OK;
 * d_action, then d_pred not NULL, objective MEAN or WORST, no d_weight with WORST, flags 0 or ABR_MPC_EXHAUSTIVE
 * (ABR_ERR_INVALID); horizon in [1, 8] and A^horizon <= 2^31 - 1, then n_scen in [1, 16] (ABR_ERR_RANGE).
 * d_best_seq rows hold -1 past h. */
int abr_env_mpc_decide_scen(AbrEnv* env, int horizon, int n_scen, int objective, int flags,
                            const double* d_pred /*[N][n_scen][horizon]*/, const double* d_weight /*[N][n_scen], nullable*/,
                            int32_t* d_action, double* d_best_j /*[N], nullable*/,
                            int32_t* d_best_seq /*[N][horizon], nullable*/, void* stream);

#ifdef __cplusplus
}
#endif
#endif
