// MPC decision kernel (SPEC.md §5): exhaustive A^h lookahead with tie-exact first-minimum.
//
// Replaces MPCBitrateController.next_bitrate (mpc.py:181-186) = predict_throughput (mpc.py:81-93) +
// scipy.optimize.brute over objective (mpc.py:120-162, buffer model mpc.py:104-118).
//
// Mapping: WPS warps (32·WPS threads) per session.
//   1. predictor: lanes invert the history samples in parallel, the harmonic sum is then accumulated
//      oldest-first in the reference's order (warp shuffles), every lane redundantly.
//   2. tables RB/DL/U[h][A] (the 2·h·A divisions the reference repeats A^h·3 times) -> shared memory.
//   3. search: the A^h sequences form a prefix tree.  All partial sums of mpc.py:144-156 after step i
//      depend only on a_0..a_i and are accumulated left to right, so carrying them down the tree executes
//      bit-identical fp64 operations to the reference's independent rollouts.  Each thread owns the
//      prefixes p = tid, tid+32·WPS, ... of depth h-2 (ascending, so its own scan order is lexicographic),
//      recomputes that prefix's state (h-2 interior steps) and then walks the last two levels fully
//      unrolled (A interior + A² leaf evaluations) with the last two table rows held in registers.
//   4. argmin: per-thread strict '<' keeps the first minimum; across threads the key (J, linear index)
//      is reduced with warp shuffles (and shared memory across warps), linear index = Σ a_i·A^(h-1-i),
//      i.e. scipy.optimize.brute's C-order first minimum (mpc.py:171-179).
//
// Bound by FP64 issue (DADD/DMUL/DSETP), not by memory: ~100 B read per decision vs ~1e5 fp64 ops.
#include "abr_common.cuh"
#include "abr_mpc_search.cuh"

namespace abr {

#ifdef ABR_MPC_COUNT   // development only: how much of the enumeration the bound leaves (abr_debug_mpc_counters)
__device__ unsigned long long g_mpc_cnt[4];   // prefixes seen, prefixes evaluated (lane level), rows evaluated, warp rounds executed
#define ABR_MPC_CNT(i, n) atomicAdd(&g_mpc_cnt[i], (unsigned long long)(n))
#else
#define ABR_MPC_CNT(i, n) do { } while (0)
#endif

namespace {

constexpr int kMaxH = 8;
constexpr int kMaxA = 16;
constexpr int kMpcWarpsPerBlock = 4;
constexpr int kPrefixCache = 64;   // parent states cached in shared memory per session (4 doubles each)
constexpr int kMaxLivePrefix = 256;  // shapes search_compact takes: A^(h-2) prefixes and A^(h-1) rows at most
constexpr int kMaxLiveRow = 1536;

// Search all A^h sequences for one session; h >= 2.  sU/sRB/sDL are [h][A] tables in shared memory,
// sAD is |U[h-1][a] - U[h-1][a']| as [a][a'] (the leaf-level smoothness term).
// AT > 0: compile-time ladder size (loops fully unrolled); AT == 0: runtime A (generic path).
// VW1: smooth_penalty == 1.0, so vw*qv == qv exactly and the multiply is dropped.
// WPS: warps per session (selects the barrier that separates filling and reading the parent-state cache).
// PRUNE (CLAMP only, penalties >= 0): branch and bound.  The value of every completion of a partial sequence is at
// most (sums so far, combined as the objective combines them) + (the best the levels still to come can add: utility
// minus the smoothness it costs, bound_tables; rebuffering still to come >= 0) — prune_bound, with a slack that dwarfs
// the rounding of the operations involved.  A prefix (or a prefix + one more level) whose bound is strictly below a
// value some sequence is known to reach cannot hold the optimum nor tie with it, and is skipped; the sequences that are
// evaluated are evaluated exactly as before, so the result — first minimum of J in C order included — is that of the
// exhaustive enumeration.  `floor_q`: a value known to be reached (the best of the constant sequences, evaluated first).
template <int AT, bool CLAMP, bool VW1, int WPS, bool PRUNE>
__device__ __forceinline__ SearchOut search(const double* __restrict__ sU, const double* __restrict__ sRB,
                                            const double* __restrict__ sDL, const double* __restrict__ sAD,
                                            double* __restrict__ sPC, const int a_rt, const int h, const int prev_q,
                                            const double buf0, const double vw, const double rw, const double L,
                                            const double B, const int tid, const int nthreads, const double floor_q,
                                            const double* __restrict__ g5, const double* __restrict__ g45) {
    constexpr bool prune = PRUNE;
    const int A = AT > 0 ? AT : a_rt;
    constexpr bool REGTAB = AT > 0 && AT <= 6;   // larger ladders keep the rows in shared memory
    constexpr int AR = REGTAB ? AT : 1;         // register-array extent
    const int P = h - 2;
    int n_prefix = 1;
    for (int i = 0; i < P; ++i) n_prefix *= A;
    const int i4 = h - 2, i5 = h - 1;
    ABR_CHECK(h >= 2 && h <= kMaxH && A >= 1 && A <= kMaxA && (prev_q < A), "search shape");
    // the leaf-level rows are uniform across threads and prefixes and read A times per prefix: keep them in registers
    double U5[AR], RB5[AR];
    if (REGTAB) {
#pragma unroll
        for (int a = 0; a < AR; ++a) { U5[a] = sU[i5 * A + a]; RB5[a] = sRB[i5 * A + a]; }
    }
    // Parent-state cache: the running sums after the first P-1 levels are shared by A prefixes each; when there are
    // few enough (36 at A = 6, h = 5) they are computed once per decision into shared memory, so a prefix costs one
    // interior step instead of P.  Same operations in the same order as the from-scratch path below.
    const int n_par = P >= 2 ? n_prefix / A : 0;
    const bool use_cache = P >= 2 && n_par <= kPrefixCache;
    if (use_cache) {
        for (int idx = tid; idx < n_par; idx += nthreads) {
            int dig[kMaxH];
            int rem = idx;
#pragma unroll
            for (int i = kMaxH - 4; i >= 0; --i) {
                if (i < P - 1) { dig[i] = rem % A; rem /= A; }
            }
            double vq = 0.0, qv = 0.0, rt = 0.0, b = buf0;
            int ap = prev_q;
#pragma unroll
            for (int i = 0; i < kMaxH - 3; ++i) {
                if (i < P - 1) {
                    const int a = dig[i];
                    const double u = sU[i * A + a];
                    const double up = ap >= 0 ? sU[i * A + ap] : u;
                    interior<CLAMP>(vq, qv, rt, b, u, fabs(dsub(u, up)), sRB[i * A + a], sDL[i * A + a], L, B);
                    ap = a;
                }
            }
            ABR_CHECK(idx >= 0 && idx < kPrefixCache, "parent-state cache slot (write)");
            sPC[idx * 4 + 0] = vq; sPC[idx * 4 + 1] = qv; sPC[idx * 4 + 2] = rt; sPC[idx * 4 + 3] = b;
        }
        if (WPS > 1) __syncthreads(); else __syncwarp();
    }
    double best_q = __longlong_as_double(0xfff0000000000000ll);  // -inf
    int best_idx = 0x7fffffff;
    double thresh = floor_q;   // a value the optimum is known to reach or exceed
    for (int p0 = 0; p0 < n_prefix; p0 += nthreads) {   // uniform trip count: the warp shares its best value per round
        if (CLAMP && prune) {
            double m = best_q;
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                const double o = __shfl_xor_sync(0xffffffffu, m, off);
                m = o > m ? o : m;
            }
            thresh = m > thresh ? m : thresh;
        }
        const int p = p0 + tid;
        if (p >= n_prefix) continue;
        ABR_MPC_CNT(0, 1);
        double vq = 0.0, qv = 0.0, rt = 0.0, b = buf0;
        int ap = prev_q;
        if (use_cache) {
            const int par = p / A, a = p - par * A;
            ABR_CHECK(par >= 0 && par < kPrefixCache && par < n_par, "parent-state cache slot (read)");
            vq = sPC[par * 4 + 0]; qv = sPC[par * 4 + 1]; rt = sPC[par * 4 + 2]; b = sPC[par * 4 + 3];
            ap = par % A;                                // last digit of the parent prefix (P >= 2)
            const int i = P - 1;
            const double u = sU[i * A + a];
            interior<CLAMP>(vq, qv, rt, b, u, fabs(dsub(u, sU[i * A + ap])), sRB[i * A + a], sDL[i * A + a], L, B);
            ap = a;
        } else {
            // decode the prefix digits (most significant first) and roll the state through levels 0..P-1
            int dig[kMaxH];
            int rem = p;
#pragma unroll
            for (int i = kMaxH - 3; i >= 0; --i) {
                if (i < P) { dig[i] = rem % A; rem /= A; }
            }
#pragma unroll
            for (int i = 0; i < kMaxH - 2; ++i) {
                if (i < P) {
                    const int a = dig[i];
                    const double u = sU[i * A + a];
                    const double up = ap >= 0 ? sU[i * A + ap] : u;
                    interior<CLAMP>(vq, qv, rt, b, u, fabs(dsub(u, up)), sRB[i * A + a], sDL[i * A + a], L, B);
                    ap = a;
                }
            }
        }
        if (CLAMP && prune && ap >= 0) {   // bound over the last two levels
            if (prune_bound<VW1>(vq, qv, rt, g45[ap], vw, rw) < thresh) continue;
        }
        ABR_MPC_CNT(1, 1);
        if ((__activemask() & ((1u << (threadIdx.x & 31)) - 1u)) == 0u) ABR_MPC_CNT(3, 1);
        const double up4 = ap >= 0 ? sU[i4 * A + ap] : 0.0;
        const int base = p * A * A;
        // a4 is a rolled loop on purpose: unrolling both levels makes ptxas keep all A*A leaves in flight
        // (~240 registers, 2 warps per scheduler); A independent leaves already cover the fp64 latency
#pragma unroll 1
        for (int a4 = 0; a4 < A; ++a4) {
            const double u4 = sU[i4 * A + a4];   // uniform address: one broadcast LDS per warp
            double vq4 = vq, qv4 = qv, rt4 = rt, b4 = b;
            interior<CLAMP>(vq4, qv4, rt4, b4, u4, ap >= 0 ? fabs(dsub(u4, up4)) : 0.0,
                            sRB[i4 * A + a4], sDL[i4 * A + a4], L, B);
            if (CLAMP && prune) {   // bound over the last level
                const double t4 = best_q > thresh ? best_q : thresh;
                if (prune_bound<VW1>(vq4, qv4, rt4, g5[a4], vw, rw) < t4) continue;
            }
            ABR_MPC_CNT(2, 1);
#pragma unroll
            for (int a5 = 0; a5 < A; ++a5) {
                const double vq5 = dadd(vq4, REGTAB ? U5[a5] : sU[i5 * A + a5]);
                const double qv5 = dadd(qv4, sAD[a5 * A + a4]);
                const double d = dsub(REGTAB ? RB5[a5] : sRB[i5 * A + a5], b4);
                const double rt5 = dadd(rt4, CLAMP ? max0(d) : d);
                const double q = dsub(dsub(vq5, VW1 ? qv5 : dmul(vw, qv5)), dmul(rw, rt5));  // J = -q, mpc.py:158-162
                if (q > best_q) { best_q = q; best_idx = base + a4 * A + a5; }  // strict: first minimum of J
            }
        }
    }
    SearchOut o; o.q = best_q; o.idx = best_idx;
    return o;
}


// Branch and bound with compaction — the search of the benchmarked shape (robust mode, A^(h-2) <= 256 prefixes).
// Measured on the benchmark's sessions, the bounds of `search` leave a fifth of the prefixes and a twentieth of the
// (prefix, next action) rows alive, but a warp that walks the prefixes lane by lane still executes a round of them as
// long as ONE of its 32 lanes survives: 3-4 of 7 rounds.  Here the survivors are compacted first (ballot + a
// shared-memory cursor), so that every round of the expensive part works on 32 live items:
//   1. every prefix: state after its last level from the parent cache, bound over the two levels to come -> live prefixes;
//   2. every (live prefix, a4): one more level, bound over the last level -> live rows;
//   3. every live row: its A leaves, with the warp's best value so far sharpening the bound from round to round.
// The lists are not in index order, so the leaves compare (value, linear index) in full: the first minimum of J in C
// order, as in the exhaustive enumeration.  States are recomputed rather than stored (one or two levels, ~60
// instructions, against 4 doubles of shared memory per item).
template <int AT, bool CLAMP, bool VW1, int WPS>
__device__ __forceinline__ SearchOut search_compact(const double* __restrict__ sU, const double* __restrict__ sRB,
                                                    const double* __restrict__ sDL, const double* __restrict__ sAD,
                                                    double* __restrict__ sPC, int* __restrict__ n_live,
                                                    uint16_t* __restrict__ live_prefix, uint16_t* __restrict__ live_row,
                                                    const double* __restrict__ g5, const double* __restrict__ g45,
                                                    const int a_rt, const int h, const int prev_q, const double buf0,
                                                    const double vw, const double rw, const double L, const double B,
                                                    const int tid, const int nthreads, const double floor_q) {
    const int A = AT > 0 ? AT : a_rt;
    const int P = h - 2;
    int n_prefix = 1;
    for (int i = 0; i < P; ++i) n_prefix *= A;
    const int n_par = n_prefix / A;
    const int i3 = P - 1, i4 = h - 2, i5 = h - 1;
    const int lane = tid & 31;
    auto barrier = [] { if (WPS > 1) __syncthreads(); else __syncwarp(); };
    // parent states (the first P-1 levels), as in search()
    if (tid < 2) n_live[tid] = 0;
    for (int idx = tid; idx < n_par; idx += nthreads) {
        int dig[kMaxH];
        int rem = idx;
#pragma unroll
        for (int i = kMaxH - 4; i >= 0; --i) {
            if (i < P - 1) { dig[i] = rem % A; rem /= A; }
        }
        double vq = 0.0, qv = 0.0, rt = 0.0, b = buf0;
        int ap = prev_q;
#pragma unroll
        for (int i = 0; i < kMaxH - 3; ++i) {
            if (i < P - 1) {
                const int a = dig[i];
                const double u = sU[i * A + a];
                const double up = ap >= 0 ? sU[i * A + ap] : u;
                interior<CLAMP>(vq, qv, rt, b, u, fabs(dsub(u, up)), sRB[i * A + a], sDL[i * A + a], L, B);
                ap = a;
            }
        }
        sPC[idx * 4 + 0] = vq; sPC[idx * 4 + 1] = qv; sPC[idx * 4 + 2] = rt; sPC[idx * 4 + 3] = b;
    }
    barrier();
    // state of prefix p after its last level (level i3) from its parent's cached state
    auto prefix_state = [&](const int p, double& vq, double& qv, double& rt, double& b) -> int {
        const int par = p / A, a = p - par * A;
        ABR_CHECK(par >= 0 && par < kPrefixCache && par < n_par, "parent-state cache slot (read)");
        vq = sPC[par * 4 + 0]; qv = sPC[par * 4 + 1]; rt = sPC[par * 4 + 2]; b = sPC[par * 4 + 3];
        const int ap = par % A;
        const double u = sU[i3 * A + a];
        interior<CLAMP>(vq, qv, rt, b, u, fabs(dsub(u, sU[i3 * A + ap])), sRB[i3 * A + a], sDL[i3 * A + a], L, B);
        return a;
    };
    // appends the items of the lanes with `live` to a list, in lane order within the warp
    auto append = [&](const bool live, const int item, uint16_t* __restrict__ list, int* __restrict__ count, const int cap) {
        const unsigned mask = __ballot_sync(0xffffffffu, live);
        if (mask == 0u) return;
        int base = 0;
        const int leader = __ffs(mask) - 1;
        if (lane == leader) base = atomicAdd(count, __popc(mask));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (live) {
            const int pos = base + __popc(mask & ((1u << lane) - 1u));
            ABR_CHECK(pos >= 0 && pos < cap, "live list slot");
            list[pos] = (uint16_t)item;
        }
    };
    // 1. live prefixes
    for (int p0 = 0; p0 < n_prefix; p0 += nthreads) {
        const int p = p0 + tid;
        bool live = false;
        if (p < n_prefix) {
            double vq, qv, rt, b;
            const int a3 = prefix_state(p, vq, qv, rt, b);
            live = !(prune_bound<VW1>(vq, qv, rt, g45[a3], vw, rw) < floor_q);
            ABR_MPC_CNT(0, 1);
        }
        append(live, p, live_prefix, &n_live[0], kMaxLivePrefix);
    }
    barrier();
    // 2. live rows: (live prefix, a4)
    const int n1 = n_live[0];
    for (int k0 = 0; k0 < n1 * A; k0 += nthreads) {
        const int k = k0 + tid;
        bool live = false;
        int row = 0;
        if (k < n1 * A) {
            const int li = k / A, a4 = k - li * A;
            const int p = live_prefix[li];
            double vq, qv, rt, b;
            const int ap = prefix_state(p, vq, qv, rt, b);
            const double u4 = sU[i4 * A + a4];
            interior<CLAMP>(vq, qv, rt, b, u4, fabs(dsub(u4, sU[i4 * A + ap])), sRB[i4 * A + a4], sDL[i4 * A + a4], L, B);
            live = !(prune_bound<VW1>(vq, qv, rt, g5[a4], vw, rw) < floor_q);
            row = p * A + a4;
            ABR_MPC_CNT(1, 1);
        }
        append(live, row, live_row, &n_live[1], kMaxLiveRow);
    }
    barrier();
    // 3. the leaves of the live rows
    const int n2 = n_live[1];
    double best_q = __longlong_as_double(0xfff0000000000000ll);  // -inf
    int best_idx = 0x7fffffff;
    double thresh = floor_q;
    for (int j0 = 0; j0 < n2; j0 += nthreads) {
        {   // the warp's best value so far
            double m = best_q;
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                const double o = __shfl_xor_sync(0xffffffffu, m, off);
                m = o > m ? o : m;
            }
            thresh = m > thresh ? m : thresh;
        }
        const int j = j0 + tid;
        if (j >= n2) continue;
        const int row = live_row[j];
        const int p = row / A, a4 = row - p * A;
        double vq4, qv4, rt4, b4;
        const int ap = prefix_state(p, vq4, qv4, rt4, b4);
        const double u4 = sU[i4 * A + a4];
        interior<CLAMP>(vq4, qv4, rt4, b4, u4, fabs(dsub(u4, sU[i4 * A + ap])), sRB[i4 * A + a4], sDL[i4 * A + a4], L, B);
        if (prune_bound<VW1>(vq4, qv4, rt4, g5[a4], vw, rw) < thresh) continue;
        ABR_MPC_CNT(2, 1);
        const int base = row * A;
#pragma unroll
        for (int a5 = 0; a5 < (AT > 0 ? AT : 1); ++a5) {
            if (AT > 0) {
                const double vq5 = dadd(vq4, sU[i5 * A + a5]);
                const double qv5 = dadd(qv4, sAD[a5 * A + a4]);
                const double d = dsub(sRB[i5 * A + a5], b4);
                const double rt5 = dadd(rt4, CLAMP ? max0(d) : d);
                const double q = dsub(dsub(vq5, VW1 ? qv5 : dmul(vw, qv5)), dmul(rw, rt5));
                if (q > best_q || (q == best_q && base + a5 < best_idx)) { best_q = q; best_idx = base + a5; }
            }
        }
        if (AT == 0) {
            for (int a5 = 0; a5 < A; ++a5) {
                const double vq5 = dadd(vq4, sU[i5 * A + a5]);
                const double qv5 = dadd(qv4, sAD[a5 * A + a4]);
                const double d = dsub(sRB[i5 * A + a5], b4);
                const double rt5 = dadd(rt4, CLAMP ? max0(d) : d);
                const double q = dsub(dsub(vq5, VW1 ? qv5 : dmul(vw, qv5)), dmul(rw, rt5));
                if (q > best_q || (q == best_q && base + a5 < best_idx)) { best_q = q; best_idx = base + a5; }
            }
        }
    }
    SearchOut o; o.q = best_q; o.idx = best_idx;
    return o;
}

// The best objective value among the A constant sequences (a, a, ..., a), lane a evaluating sequence a with exactly
// the operations the search performs for it: a value the optimum reaches or exceeds, known before the search starts.
template <bool CLAMP, bool VW1>
__device__ __forceinline__ double probe_constant(const double* __restrict__ sU, const double* __restrict__ sRB,
                                                 const double* __restrict__ sDL, const int A, const int h,
                                                 const int prev_q, const double buf0, const double vw, const double rw,
                                                 const double L, const double B, const int lane) {
    double q = __longlong_as_double(0xfff0000000000000ll);  // -inf
    if (lane < A) {
        const int a = lane;
        double vq = 0.0, qv = 0.0, rt = 0.0, b = buf0;
        int ap = prev_q;
        for (int i = 0; i < h - 1; ++i) {
            const double u = sU[i * A + a];
            const double up = ap >= 0 ? sU[i * A + ap] : u;
            interior<CLAMP>(vq, qv, rt, b, u, fabs(dsub(u, up)), sRB[i * A + a], sDL[i * A + a], L, B);
            ap = a;
        }
        const int i5 = h - 1;
        const double u5 = sU[i5 * A + a];
        const double vq5 = dadd(vq, u5);
        const double qv5 = dadd(qv, ap >= 0 ? fabs(dsub(u5, sU[i5 * A + ap])) : 0.0);
        const double d = dsub(sRB[i5 * A + a], b);
        const double rt5 = dadd(rt, CLAMP ? max0(d) : d);
        q = dsub(dsub(vq5, VW1 ? qv5 : dmul(vw, qv5)), dmul(rw, rt5));
        if (!(q == q)) q = __longlong_as_double(0xfff0000000000000ll);   // a NaN bounds nothing
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const double o = __shfl_xor_sync(0xffffffffu, q, off);
        q = o > q ? o : q;
    }
    return q;
}

struct __align__(8) SessShared {
    double U[kMaxH * kMaxA], RB[kMaxH * kMaxA], DL[kMaxH * kMaxA], AD[kMaxA * kMaxA];
    double PC[kPrefixCache * 4];
    double redq[kMpcWarpsPerBlock];
    int redi[kMpcWarpsPerBlock];
};
// branch and bound with compaction (search_compact): the prefixes, then the (prefix, next action) rows that survive
// their bounds, and how many there are.  Only the pruning kernels carry the lists.
template <bool PRUNE>
struct LiveLists {
    int n_live[2];
    uint16_t live_prefix[PRUNE ? kMaxLivePrefix : 2];
    uint16_t live_row[PRUNE ? kMaxLiveRow : 2];
    double g5[PRUNE ? kMaxA : 1], g45[PRUNE ? kMaxA : 1];   // best that the last level / the last two levels can still add
};

// WPS warps per session; blockDim.x = 32 * kMpcWarpsPerBlock; sessions per block = kMpcWarpsPerBlock / WPS.
// AT = compile-time ladder size (0 = runtime A), CLAMP = robust mode (SPEC §5.2) — one kernel per shape so
// that each gets its own register allocation.
// PRUNE (with CLAMP): branch and bound (search / search_compact); decided by the host (robust mode, non-negative
// penalties, no ABR_MPC_EXHAUSTIVE).  A template parameter so that the enumerating kernel carries none of it.
// EXT (with CLAMP, SPEC §5.6): the step-i tables divide by the caller's prediction a.pred[s][i] instead of the robust
// prediction; the history ring and the robust state are neither read nor written.  Everything from the tables on is
// the robust search: it reads only the per-step tables, and the bounds of branch and bound only U.
#ifndef ABR_MPC_PRUNE_BLOCKS
#define ABR_MPC_PRUNE_BLOCKS 5
#endif
template <int WPS, int AT, bool CLAMP, bool PRUNE, bool EXT = false>
__global__ void __launch_bounds__(32 * kMpcWarpsPerBlock, PRUNE ? ABR_MPC_PRUNE_BLOCKS : 5)   // <= 96 registers: 20 warps per SM (A/B-tested: 4 -> 5 +3 %, 6 -3 %)
abr_mpc_kernel(const MpcArgs a) {
    static_assert(!EXT || CLAMP, "caller predictions use the robust objective");
    constexpr int SPB = kMpcWarpsPerBlock / WPS;
    __shared__ SessShared sh[SPB];
    __shared__ LiveLists<PRUNE> live[SPB];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int slot = warp / WPS;                 // session slot inside the block
    const int wis = warp % WPS;                  // warp index inside the session
    const int tid = wis * 32 + lane;             // thread index inside the session
    constexpr int NT = 32 * WPS;
    SessShared& S = sh[slot];
    LiveLists<PRUNE>& LL = live[slot];
    const AbrParams& p = a.p;
    const int A = AT > 0 ? AT : a.A, H = a.H, K = a.K;
    const double L = p.chunk_length, B = p.max_buffer;

    for (long long s = (long long)blockIdx.x * SPB + slot; s < a.N; s += (long long)gridDim.x * SPB) {
        // Every thread of a session computes the quantities below redundantly and identically, so control flow
        // (and, for WPS > 1 where one block serves one session, every __syncthreads) is uniform.
        const int k = a.chunk_idx[s];
        const int prev_q = a.prev_q[s];
        const double buf0 = a.buffer[s];
        const int hlen = EXT ? 0 : a.hist_len[s];   // EXT: no history (the call works without track_history)
        const int n = hlen < K ? hlen : K;
        const int start = hlen <= K ? 0 : hlen % K;
        const bool inert = a.done && a.done[s];
        int h = H;
        int status = 0;  // 0 search, 1 fixed action (act), 2 error
        int act = -1;
        if (inert) { status = 1; act = 0; }
        else if (k < 0 || prev_q >= A) status = 2;
        else if (!EXT && n <= 0) {
            if (a.mode == ABR_MPC_ROBUST || (a.flags & ABR_MPC_EMPTY_DEFAULT)) { status = 1; act = p.default_quality > 0 ? p.default_quality : 0; }
            else status = 2;                                               // ZeroDivisionError, mpc.py:90
        }
        if (status == 0) {
            if (k + H > a.V) {
                if (a.mode == ABR_MPC_ROBUST || (a.flags & ABR_MPC_TRUNCATE)) h = a.V - k;
                else status = 2;                                           // IndexError, mpc.py:125-128
                if (status == 0 && h <= 0) { status = 1; act = 0; }
            }
        }
        if constexpr (EXT) {
            if (status == 0) {
                // ---- caller predictions (SPEC §5.6): lane i < h reads p_i; one that is not finite and > 0 is an input
                //      error.  Every warp of the session reads them, so status stays uniform across the session. ----
                double pv = 1.0;
                if (lane < h) pv = a.pred[s * H + lane];
                if (__ballot_sync(0xffffffffu, lane < h && !(pv > 0.0 && pv < __longlong_as_double(0x7ff0000000000000ll))) != 0u)
                    status = 2;
                else {
                    for (int e = tid; e < h * A; e += NT) {   // the robust branch's fill, with p_i for c_rob
                        ABR_CHECK(e < kMaxH * kMaxA && (k + e / A) < a.V, "lookahead table entry");
                        const int i = e / A, aa = e - i * A;
                        const double dl = ddiv(a.sizes[(k + i) * A + aa], a.pred[s * H + i]);
                        S.RB[e] = dl; S.DL[e] = dl;
                        S.U[e] = a.util[(k + i) * A + aa];
                    }
                }
            }
        }
        double c_rob = 0.0;
        if (!EXT && status == 0) {
            // ---- predictor: S = sum of 1/x oldest first (mpc.py:84-88) ----
            double Ssum = 0.0;
            bool bad = false;
            double newest = 0.0;
            for (int j0 = 0; j0 < n; j0 += 32) {
                const int j = j0 + lane;
                double x = 1.0;
                if (j < n) x = a.bw_hist[s * a.hist_session_stride + (long long)((start + j) % K) * a.hist_slot_stride];
                const bool xbad = (a.mode == ABR_MPC_REF) ? (x == 0.0) : !(x > 0.0);
                bad |= (__ballot_sync(0xffffffffu, xbad && j < n) != 0u);
                const double inv = ddiv(1.0, x);
                const int m = min(32, n - j0);
                for (int jj = 0; jj < m; ++jj) Ssum = dadd(Ssum, __shfl_sync(0xffffffffu, inv, jj));
                if (j0 + 32 >= n) newest = __shfl_sync(0xffffffffu, x, m - 1);
            }
            // ---- predictor "expsmoothing" (mpc.py:72-79; SPEC §5.4): flat forecast l_n of simple exponential
            //      smoothing with alpha = 0.5 and the least-squares initial level; sequential, every thread redundantly ----
            double ses = 0.0;
            const bool use_ses = a.mode == ABR_MPC_REF && (a.flags & ABR_MPC_PRED_SES) != 0;
            if (use_ses && !bad) {
                double la = 0.0, lb = 1.0, num = 0.0, den = 0.0;          // l_t = la + lb * l_0
                for (int j = 0; j < n; ++j) {
                    const double y = a.bw_hist[s * a.hist_session_stride + (long long)((start + j) % K) * a.hist_slot_stride];
                    const double r = dsub(y, la);                           // one-step error with l_0 = 0
                    num = dadd(num, dmul(lb, r));
                    den = dadd(den, dmul(lb, lb));
                    la = dadd(dmul(0.5, y), dmul(0.5, la));
                    lb = dmul(0.5, lb);
                }
                ses = dadd(la, dmul(lb, ddiv(num, den)));
                if (!(ses > 0.0)) bad = true;                               // a non-positive forecast cannot be divided by
            }
            if (bad) status = 2;                                           // ZeroDivisionError, mpc.py:88
            else if (a.mode == ABR_MPC_REF) {
                // p_i = (n+i)/S ; S += 1/p_i   (mpc.py:83-92 incl. the list mutation D10)
                for (int i = 0; i < h; ++i) {
                    const double pi = use_ses ? ses : ddiv((double)(n + i), Ssum);
                    Ssum = dadd(Ssum, ddiv(1.0, pi));
                    if (a.preds && tid == 0) a.preds[s * H + i] = pi;
                    // tables for step i: each thread of the session fills entries a = tid, tid+NT, ...
                    for (int aa = tid; aa < A; aa += NT) {
                        ABR_CHECK(i * A + aa < kMaxH * kMaxA && k + i < a.V, "lookahead table entry");
                        const double sz = a.sizes[(k + i) * A + aa];
                        double m = sz > 0.0 ? sz : 0.0;                    // max(0, size, L), mpc.py:151 (D11)
                        if (L > m) m = L;
                        S.RB[i * A + aa] = ddiv(m, pi);
                        S.DL[i * A + aa] = ddiv(a.sizes[k * A + aa], pi);  // D12: chunk k's sizes
                        S.U[i * A + aa] = a.util[(k + i) * A + aa];
                    }
                }
            } else {
                const double hm = ddiv((double)n, Ssum);
                double max_err = 0.0;
                if (a.last_pred) {
                    const double lp = a.last_pred[s];
                    int el = a.err_len[s];
                    double* ring = a.err_ring + s * a.hist_session_stride;
                    double e_new = 0.0;
                    const bool push = lp > 0.0;
                    if (push) e_new = ddiv(fabs(dsub(lp, newest)), newest);
                    const int slot_new = el % K;
                    const int m = (el + (push ? 1 : 0)) < K ? (el + (push ? 1 : 0)) : K;
                    for (int j = 0; j < m; ++j) {
                        const double e = (push && j == slot_new) ? e_new : ring[(long long)j * a.hist_slot_stride];
                        if (e > max_err) max_err = e;
                    }
                    __syncwarp();
                    if (WPS > 1) __syncthreads();   // every thread has read the old state before it is replaced
                    if (tid == 0) {
                        if (push) { ring[(long long)slot_new * a.hist_slot_stride] = e_new; a.err_len[s] = el + 1; }
                        a.last_pred[s] = hm;
                    }
                }
                c_rob = ddiv(hm, dadd(1.0, max_err));
                if (a.preds && tid < H) a.preds[s * H + tid] = c_rob;
                for (int e = tid; e < h * A; e += NT) {
                    ABR_CHECK(e < kMaxH * kMaxA && (k + e / A) < a.V, "lookahead table entry");
                    const int i = e / A, aa = e - i * A;
                    const double dl = ddiv(a.sizes[(k + i) * A + aa], c_rob);
                    S.RB[e] = dl; S.DL[e] = dl;
                    S.U[e] = a.util[(k + i) * A + aa];
                }
            }
        }
        // NOTE: status is identical in every thread of the session (all inputs are session-uniform).
        if (WPS > 1) __syncthreads(); else __syncwarp();
        SearchOut o; o.q = 0.0; o.idx = 0;
        double ts_best = 0.0;
        if (status == 0) {
            const int i5 = h - 1;
            for (int e = tid; e < A * A; e += NT) {
                const int a5 = e / A, a4 = e - a5 * A;
                S.AD[e] = fabs(dsub(S.U[i5 * A + a5], S.U[i5 * A + a4]));
            }
            if (WPS > 1) __syncthreads(); else __syncwarp();
            // Start-up phase (SPEC §5.3; f_st of mpc.py:7-18, the TODO of mpc.py:141): the start-up delay T_s is a second
            // decision variable on the grid jt * ts_step; it is credited to the initial buffer and charged
            // startup_weight * T_s (mpc.py:160).  T_s is the slowest axis of the enumeration: ties keep the smaller T_s.
            const int n_ts = (a.n_ts > 1 && (!a.startup || a.startup[s])) ? a.n_ts : 1;   // session-uniform
            double q_best = __longlong_as_double(0xfff0000000000000ll);
            int idx_best = 0x7fffffff;
            for (int jt = 0; jt < n_ts; ++jt) {
                const double ts = jt == 0 ? 0.0 : dmul((double)jt, a.ts_step);
                const double bufj = jt == 0 ? buf0 : dadd(buf0, ts);
                if (h == 1) {
                    // single level: A leaves, thread 0 of the session scans them in order
                    double bq = __longlong_as_double(0xfff0000000000000ll);
                    int bi = 0x7fffffff;
                    if (tid == 0) {
                        for (int a0 = 0; a0 < A; ++a0) {
                            const double u = S.U[a0];
                            const double qv = prev_q >= 0 ? fabs(dsub(u, S.U[prev_q])) : 0.0;
                            const double d = dsub(S.RB[a0], bufj);
                            const double rt = CLAMP ? max0(d) : d;
                            // 0 + x is exact, so the running sums of mpc.py:146-152 reduce to the terms themselves
                            const double q = dsub(dsub(u, dmul(p.smooth_penalty, qv)), dmul(p.rebuf_penalty, rt));
                            if (q > bq) { bq = q; bi = a0; }
                        }
                    }
                    o.q = bq; o.idx = bi;
                } else {
                    const double ninf = __longlong_as_double(0xfff0000000000000ll);
                    // the compacted form: shapes with a parent cache whose prefixes and rows fit the lists
                    int n_pre = 1;
                    for (int i = 0; i < h - 2; ++i) n_pre *= A;
                    const bool compact = PRUNE && h >= 4 && n_pre / A <= kPrefixCache && n_pre <= kMaxLivePrefix &&
                                         n_pre * A <= kMaxLiveRow;
                    if (PRUNE) {
                        bound_tables(S.U, A, h, p.smooth_penalty, LL.g5, LL.g45, lane);
                        if (WPS > 1) __syncthreads();
                    }
                    if (p.smooth_penalty == 1.0) {
                        const double fl = PRUNE ? probe_constant<CLAMP, true>(S.U, S.RB, S.DL, A, h, prev_q, bufj, 1.0,
                                                                              p.rebuf_penalty, L, B, lane) : ninf;
                        if (PRUNE && compact)
                            o = search_compact<AT, CLAMP, true, WPS>(S.U, S.RB, S.DL, S.AD, S.PC, LL.n_live, LL.live_prefix, LL.live_row, LL.g5, LL.g45,
                                                                     A, h, prev_q, bufj, 1.0, p.rebuf_penalty, L, B, tid, NT, fl);
                        else
                            o = search<AT, CLAMP, true, WPS, PRUNE>(S.U, S.RB, S.DL, S.AD, S.PC, A, h, prev_q, bufj, 1.0,
                                                                    p.rebuf_penalty, L, B, tid, NT, fl, LL.g5, LL.g45);
                    } else {
                        const double fl = PRUNE ? probe_constant<CLAMP, false>(S.U, S.RB, S.DL, A, h, prev_q, bufj,
                                                                               p.smooth_penalty, p.rebuf_penalty, L, B, lane) : ninf;
                        if (PRUNE && compact)
                            o = search_compact<AT, CLAMP, false, WPS>(S.U, S.RB, S.DL, S.AD, S.PC, LL.n_live, LL.live_prefix, LL.live_row, LL.g5, LL.g45,
                                                                      A, h, prev_q, bufj, p.smooth_penalty, p.rebuf_penalty, L, B, tid,
                                                                      NT, fl);
                        else
                            o = search<AT, CLAMP, false, WPS, PRUNE>(S.U, S.RB, S.DL, S.AD, S.PC, A, h, prev_q, bufj, p.smooth_penalty,
                                                                     p.rebuf_penalty, L, B, tid, NT, fl, LL.g5, LL.g45);
                    }
                }
                // ---- argmin over the session's threads: key (J, linear index) ----
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) {
                    const double oq = __shfl_xor_sync(0xffffffffu, o.q, off);
                    const int oi = __shfl_xor_sync(0xffffffffu, o.idx, off);
                    better(o.q, o.idx, oq, oi);
                }
                if (WPS > 1) {
                    if (lane == 0) { S.redq[wis] = o.q; S.redi[wis] = o.idx; }
                    __syncthreads();
                    o.q = S.redq[0]; o.idx = S.redi[0];
                    for (int w = 1; w < WPS; ++w) better(o.q, o.idx, S.redq[w], S.redi[w]);
                }
                if (n_ts == 1) break;                                  // the usual decision: nothing else to do
                // every thread of the session holds the same reduced (q, idx): the comparison below is uniform
                const double qt = dsub(o.q, dmul(p.startup_penalty, ts));
                if (qt > q_best) { q_best = qt; idx_best = o.idx; ts_best = ts; }
                if (WPS > 1) __syncthreads(); else __syncwarp();       // the parent-state cache / redq are reused
            }
            if (n_ts > 1) { o.q = q_best; o.idx = idx_best; }
        }
        if (tid == 0) {
            if (status == 0) {
                int idx = o.idx == 0x7fffffff ? 0 : o.idx;   // all scores -inf/NaN: first sequence
                int div = 1, first = idx;            // first action = idx / A^(h-1): h-1 divisions by A (a constant
                for (int i = 1; i < h; ++i) { div *= A; first /= A; }   // when the ladder size is a template argument)
                a.action[s] = first;
                if (a.startup_delay) a.startup_delay[s] = ts_best;
                if (a.best_j) a.best_j[s] = -o.q;
                if (a.best_seq) {
                    int rem = idx, d = div;
                    for (int i = 0; i < H; ++i) {
                        if (i < h) { a.best_seq[s * H + i] = rem / d; rem %= d; d = d > 1 ? d / A : 1; }
                        else a.best_seq[s * H + i] = -1;
                    }
                }
            } else {
                a.action[s] = status == 1 ? act : -1;
                if (a.startup_delay) a.startup_delay[s] = 0.0;
                if (a.best_j) a.best_j[s] = __longlong_as_double(0x7ff8000000000000ll);
                if (a.best_seq) for (int i = 0; i < H; ++i) a.best_seq[s * H + i] = -1;
                if (a.preds && status == 2) for (int i = 0; i < H; ++i) a.preds[s * H + i] = 0.0;
                if (status == 2) {
                    if (a.error_count64) atomicAdd(a.error_count64, 1ull);
                    if (a.error_count32) atomicAdd(a.error_count32, 1);
                }
            }
        }
        if (WPS > 1) __syncthreads(); else __syncwarp();  // tables are reused by the next session of this slot
    }
}

// ---- objective() of given sequences (mpc.py:120-162): one thread per sequence, each rolled out independently
//      from scratch exactly like the reference does.  Used by MPCBitrateController.objective and by the parity
//      tests that compare the whole score grid against the reference's. ----
__global__ void __launch_bounds__(128)
abr_mpc_score_kernel(const double* __restrict__ sizes, const double* __restrict__ util, int V, int A, AbrParams p,
                     int k, int prev_q, double buffer, const double* __restrict__ hist, int n, int H, int mode,
                     double max_err, const int32_t* __restrict__ seqs, int M, double* __restrict__ scores) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= M) return;
    const double L = p.chunk_length, B = p.max_buffer;
    double S = 0.0;
    for (int j = 0; j < n; ++j) S = dadd(S, ddiv(1.0, hist[j]));
    const double c = mode == ABR_MPC_ROBUST ? ddiv(ddiv((double)n, S), dadd(1.0, max_err)) : 0.0;
    double vq = 0.0, qv = 0.0, rt = 0.0, b = buffer;
    int ap = prev_q;
    for (int i = 0; i < H; ++i) {
        const int a = seqs[(size_t)m * H + i];
        double pi = c;
        if (mode == ABR_MPC_REF) { pi = ddiv((double)(n + i), S); S = dadd(S, ddiv(1.0, pi)); }
        const double u = util[(k + i) * A + a];
        vq = dadd(vq, u);
        if (ap >= 0) qv = dadd(qv, fabs(dsub(u, util[(k + i) * A + ap])));
        double d, dl;
        if (mode == ABR_MPC_REF) {
            const double sz = sizes[(k + i) * A + a];
            double mx = sz > 0.0 ? sz : 0.0;
            if (L > mx) mx = L;
            d = dsub(ddiv(mx, pi), b);
            dl = ddiv(sizes[k * A + a], pi);
        } else {
            dl = ddiv(sizes[(k + i) * A + a], pi);
            d = max0(dsub(dl, b));
        }
        rt = dadd(rt, d);
        if (i != H - 1) {
            const double t = max0(dsub(b, dl));
            const double tl = dadd(t, L);
            const double w = max0(dsub(tl, B));
            b = max0(dsub(tl, w));
        }
        ap = a;
    }
    scores[m] = -dsub(dsub(vq, dmul(p.smooth_penalty, qv)), dmul(p.rebuf_penalty, rt));
}

// ---- FP64 issue-rate probe (roofline denominator of the MPC kernel) ----
template <int KIND>
__global__ void __launch_bounds__(256) abr_fp64_probe_kernel(int iters, double* sink) {
    double x0 = 1.0 + threadIdx.x * 1e-9, x1 = x0 + 1e-3, x2 = x0 + 2e-3, x3 = x0 + 3e-3;
    double x4 = x0 + 4e-3, x5 = x0 + 5e-3, x6 = x0 + 6e-3, x7 = x0 + 7e-3;
    const double c = 1.0000001, d = 1e-7;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            if (KIND == 0) {        // 8 independent DADD chains
                x0 = dadd(x0, d); x1 = dadd(x1, d); x2 = dadd(x2, d); x3 = dadd(x3, d);
                x4 = dadd(x4, d); x5 = dadd(x5, d); x6 = dadd(x6, d); x7 = dadd(x7, d);
            } else if (KIND == 1) { // 8 independent DFMA chains
                x0 = __fma_rn(x0, c, d); x1 = __fma_rn(x1, c, d); x2 = __fma_rn(x2, c, d); x3 = __fma_rn(x3, c, d);
                x4 = __fma_rn(x4, c, d); x5 = __fma_rn(x5, c, d); x6 = __fma_rn(x6, c, d); x7 = __fma_rn(x7, c, d);
            } else {                // DADD + DMUL + compare/select mix (4 + 2 + 2 fp64-pipe ops)
                x0 = dadd(x0, d); x1 = dmul(x1, c); x2 = dadd(x2, x0); x3 = dadd(x3, d);
                x4 = dmul(x4, c); x5 = dadd(x5, d);
                if (x2 > x6) x6 = x2;
                if (x3 > x7) x7 = x3;
            }
        }
    }
    sink[blockIdx.x * blockDim.x + threadIdx.x] = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
}

// single dependent chain per thread, one warp per SM: cycles per instruction = pipeline latency
template <int KIND>
__global__ void __launch_bounds__(32) abr_fp64_latency_kernel(int iters, double* sink, long long* cycles) {
    double x = 1.0 + threadIdx.x * 1e-9;
    const double d = 1e-7, c = 1.0000001;
    const long long t0 = clock64();
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int r = 0; r < 64; ++r) {
            if (KIND == 0) x = dadd(x, d);
            else if (KIND == 1) x = dmul(x, c);
            else x = max0(dsub(x, d));     // DADD + integer sign-mask
        }
    }
    const long long t1 = clock64();
    sink[blockIdx.x * 32 + threadIdx.x] = x;
    if (threadIdx.x == 0) cycles[blockIdx.x] = t1 - t0;
}

}  // namespace

#ifdef ABR_MPC_COUNT
}  // namespace abr
extern "C" int abr_debug_mpc_counters(unsigned long long* out, int reset) {
    cudaDeviceSynchronize();
    if (out) cudaMemcpyFromSymbol(out, abr::g_mpc_cnt, sizeof(unsigned long long) * 4);
    if (reset) { unsigned long long z[4] = {0, 0, 0, 0}; cudaMemcpyToSymbol(abr::g_mpc_cnt, z, sizeof(z)); }
    return 0;
}
namespace abr {
#endif

cudaError_t launch_fp64_latency(int kind, int iters, double* d_sink, long long* d_cycles, cudaStream_t st) {
    switch (kind) {
        case 0: abr_fp64_latency_kernel<0><<<1, 32, 0, st>>>(iters, d_sink, d_cycles); break;
        case 1: abr_fp64_latency_kernel<1><<<1, 32, 0, st>>>(iters, d_sink, d_cycles); break;
        default: abr_fp64_latency_kernel<2><<<1, 32, 0, st>>>(iters, d_sink, d_cycles); break;
    }
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_mpc(const MpcArgs& a, cudaStream_t st) {
    if (a.N <= 0) return cudaSuccess;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    // threads per session: one warp when there are enough sessions to fill the GPU, otherwise a whole block
    long long combos = 1;
    for (int i = 0; i < a.H; ++i) combos *= a.A;
    const long long warps_needed_full = (long long)sms * 16;
    const int wps = (a.N >= warps_needed_full || combos < 32 * 36 * 4) ? 1 : kMpcWarpsPerBlock;
    const int spb = kMpcWarpsPerBlock / wps;
    long long blocks = (a.N + spb - 1) / spb;
    const long long max_blocks = (long long)sms * 64;
    if (blocks > max_blocks) blocks = max_blocks;
    const bool clamp = a.mode == ABR_MPC_ROBUST;
    // branch and bound (SPEC §5.5): robust mode, non-negative penalties, unless the caller asks for the enumeration
    const bool prune = clamp && !(a.flags & ABR_MPC_EXHAUSTIVE) && a.p.smooth_penalty >= 0.0 && a.p.rebuf_penalty >= 0.0;
    const bool ext = a.pred != nullptr;   // caller predictions (SPEC §5.6): robust mode only, checked by the C-ABI
    const unsigned g = (unsigned)blocks, t = 32 * kMpcWarpsPerBlock;
#define ABR_MPC_LAUNCH(AT_)                                                                        \
    do {                                                                                           \
        if (wps == 1) {                                                                            \
            if (ext && prune) abr_mpc_kernel<1, AT_, true, true, true><<<g, t, 0, st>>>(a);        \
            else if (ext) abr_mpc_kernel<1, AT_, true, false, true><<<g, t, 0, st>>>(a);           \
            else if (prune) abr_mpc_kernel<1, AT_, true, true><<<g, t, 0, st>>>(a);                \
            else if (clamp) abr_mpc_kernel<1, AT_, true, false><<<g, t, 0, st>>>(a);               \
            else abr_mpc_kernel<1, AT_, false, false><<<g, t, 0, st>>>(a);                         \
        } else {                                                                                   \
            if (ext && prune) abr_mpc_kernel<kMpcWarpsPerBlock, AT_, true, true, true><<<g, t, 0, st>>>(a); \
            else if (ext) abr_mpc_kernel<kMpcWarpsPerBlock, AT_, true, false, true><<<g, t, 0, st>>>(a); \
            else if (prune) abr_mpc_kernel<kMpcWarpsPerBlock, AT_, true, true><<<g, t, 0, st>>>(a);     \
            else if (clamp) abr_mpc_kernel<kMpcWarpsPerBlock, AT_, true, false><<<g, t, 0, st>>>(a); \
            else abr_mpc_kernel<kMpcWarpsPerBlock, AT_, false, false><<<g, t, 0, st>>>(a);         \
        }                                                                                          \
    } while (0)
    switch (a.A) {
        case 2: ABR_MPC_LAUNCH(2); break;
        case 3: ABR_MPC_LAUNCH(3); break;
        case 4: ABR_MPC_LAUNCH(4); break;
        case 5: ABR_MPC_LAUNCH(5); break;
        case 6: ABR_MPC_LAUNCH(6); break;
        case 8: ABR_MPC_LAUNCH(8); break;
        default: ABR_MPC_LAUNCH(0); break;
    }
#undef ABR_MPC_LAUNCH
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_mpc_score(const double* d_sizes, const double* d_util, int V, int A, const AbrParams& p, int k,
                             int prev_q, double buffer, const double* d_hist, int n, int H, int mode, double max_err,
                             const int32_t* d_seqs, int M, double* d_scores, cudaStream_t st) {
    if (M <= 0) return cudaSuccess;
    abr_mpc_score_kernel<<<(M + 127) / 128, 128, 0, st>>>(d_sizes, d_util, V, A, p, k, prev_q, buffer, d_hist, n, H,
                                                          mode, max_err, d_seqs, M, d_scores);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_fp64_probe(int kind, int iters, double* d_sink, int* threads_total, long long* ops_per_thread,
                              cudaStream_t st) {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int blocks = sms * 8, threads = 256;
    *threads_total = blocks * threads;
    *ops_per_thread = (long long)iters * 64;
    switch (kind) {
        case 0: abr_fp64_probe_kernel<0><<<blocks, threads, 0, st>>>(iters, d_sink); break;
        case 1: abr_fp64_probe_kernel<1><<<blocks, threads, 0, st>>>(iters, d_sink); break;
        case 2: abr_fp64_probe_kernel<2><<<blocks, threads, 0, st>>>(iters, d_sink); break;
        default: return cudaErrorInvalidValue;
    }
    count_launch();
    return cudaGetLastError();
}

}  // namespace abr
