// MPC over caller-supplied throughput scenarios (SPEC §5.7): one search kernel, abr_mpc_scen_kernel.
//
// The per-node state grows from the 4 doubles of abr_mpc_kernel to 2 + 2K (vq and qv, which do not depend on the
// scenario, and rt_k, b_k per scenario), so this kernel has its own layout.  It shares the interior step, the
// branch-and-bound bound and the argmin comparison with abr_mpc.cu (abr_mpc_search.cuh).
//
// Mapping: warps per session by the rule of launch_mpc (one warp when there are enough sessions to fill the GPU,
// otherwise a 128-thread block).  Tables in dynamic shared memory, sized by the call: U[h][A], RB_k[h][A] per scenario,
// the leaf smoothness AD[A][A] and the weights.  A thread owns prefixes of depth h-2 (ascending, so its own scan is
// lexicographic), rolls each prefix once per scenario into a private scratch in shared memory, then walks the last two
// levels: for every a4, the child state of scenario k is one interior step from the scratch, and the A leaves below
// it take their scenario-k values from it.  Scenarios are the outer loop of the leaves, so each leaf's aggregate is
// formed in k order in registers.  Argmin: strict '>' per thread, then the (Q, linear index) reduction.
#include "abr_common.cuh"
#include "abr_mpc_search.cuh"
#include "../../include/abr_b200_mpc_scen.h"

namespace abr {
namespace {

constexpr int kScenMaxH = 8;
constexpr int kScenWarpsPerBlock = 4;   // as abr_mpc_kernel: 128 threads, 4 / WPS sessions per block
constexpr int kScenLeafChunk = 4;    // leaves per register block of the runtime-A form
constexpr int kScenThreads = 32 * kScenWarpsPerBlock;

// Doubles of shared memory per session slot: U[H][A], RB[K][H][A], AD[A][A], W[K], g5[A], g45[A], and the cross-warp
// reduction (values, then indices stored as ints in the same number of doubles).  The block adds the threads'
// scratch, [2K][kScenThreads]: rt_k and b_k of each thread's current prefix.
__host__ __device__ __forceinline__ int scen_slot_doubles(const int A, const int H, const int K) {
    return H * A + K * H * A + A * A + K + 2 * A + 2 * kScenWarpsPerBlock;
}

// Upper bound of the aggregate Q of every completion of a node (vq, qv, rt_of(k)), g the best the levels still to come
// can add.  WORST: Q <= q_k for every k, so the bound of one scenario is a bound; the one with the largest rt_k is the
// lowest.  MEAN: the weights are >= 0, so sum w_k b_k bounds sum w_k q_k in real arithmetic; 1e-9 of sum |w_k b_k|
// covers the rounding of both K-term weighted sums (at most 2 * 16 * 2^-53 of it) many times over.
template <int OBJ, typename RT>
__device__ __forceinline__ double scen_bound(const double vq, const double qv, const RT& rt_of, const int K,
                                             const double* __restrict__ sW, const double g, const double vw,
                                             const double rw) {
    if (OBJ == ABR_MPC_SCEN_WORST) {
        double m = rt_of(0);
        for (int k = 1; k < K; ++k) { const double r = rt_of(k); m = r > m ? r : m; }
        return prune_bound<false>(vq, qv, m, g, vw, rw);
    } else {
        double s = 0.0, mag = 0.0;
        for (int k = 0; k < K; ++k) {
            const double t = dmul(sW[k], prune_bound<false>(vq, qv, rt_of(k), g, vw, rw));
            s = k == 0 ? t : dadd(s, t);
            mag = dadd(mag, fabs(t));
        }
        return dadd(s, dmul(1e-9, dadd(mag, 1.0)));
    }
}

// Search all A^h sequences of one session over K scenarios.  sRB is [K][H][A]; sAD[a5 * A + a] = |U5[a5] - U5[a]|.
// `ps`: the thread's scratch (rt_k at ps[2k * kScenThreads], b_k at ps[(2k + 1) * kScenThreads]).
// PRUNE: branch and bound as in search(), with scen_bound; the warp's best value so far is the threshold.
template <int AT, int OBJ, bool PRUNE>
__device__ __forceinline__ SearchOut scen_search(const double* __restrict__ sU, const double* __restrict__ sRB,
                                                 const double* __restrict__ sAD, const double* __restrict__ sW,
                                                 const double* __restrict__ g5, const double* __restrict__ g45,
                                                 double* __restrict__ ps, const int a_rt, const int H, const int K,
                                                 const int h, const int prev_q, const double buf0, const double vw,
                                                 const double rw, const double L, const double B, const int tid,
                                                 const int nthreads) {
    const int A = AT > 0 ? AT : a_rt;
    constexpr int CH = AT > 0 ? AT : kScenLeafChunk;
    const int P = h >= 2 ? h - 2 : 0;
    int n_prefix = 1;
    for (int i = 0; i < P; ++i) n_prefix *= A;
    const int i4 = h - 2, i5 = h - 1;
    ABR_CHECK(h >= 1 && h <= kScenMaxH && A >= 1 && A <= 16 && K >= 1 && K <= ABR_MPC_SCEN_MAX && prev_q < A, "scenario search shape");
    double best_q = __longlong_as_double(0xfff0000000000000ll);  // -inf
    int best_idx = 0x7fffffff;
    // The leaves below a node after level h-2 (vq4, qv4; a4 < 0: the root of h = 1 with no previous action), whose
    // scenario-k state child(k, rt, b) gives; `base` is the linear index of leaf 0.
    auto leaves = [&](const double vq4, const double qv4, const int a4, const int base, const auto& child) {
        for (int c0 = 0; c0 < A; c0 += CH) {
            double val[CH], Q[CH];
#pragma unroll
            for (int j = 0; j < CH; ++j) {
                const int a5 = AT > 0 ? j : min(c0 + j, A - 1);
                const double vq5 = dadd(vq4, sU[i5 * A + a5]);
                const double qv5 = a4 >= 0 ? dadd(qv4, sAD[a5 * A + a4]) : qv4;
                val[j] = dsub(vq5, dmul(vw, qv5));
                Q[j] = 0.0;
            }
            for (int k = 0; k < K; ++k) {
                double rt, b;
                child(k, rt, b);
                const double w = OBJ == ABR_MPC_SCEN_MEAN ? sW[k] : 0.0;
                const double* rb = sRB + (k * H + i5) * A;
#pragma unroll
                for (int j = 0; j < CH; ++j) {
                    const int a5 = AT > 0 ? j : min(c0 + j, A - 1);
                    const double q = dsub(val[j], dmul(rw, dadd(rt, max0(dsub(rb[a5], b)))));  // q_k = (vq - vw qv) - rw rt_k
                    if (OBJ == ABR_MPC_SCEN_MEAN) {
                        const double t = dmul(w, q);
                        Q[j] = k == 0 ? t : dadd(Q[j], t);
                    } else {
                        Q[j] = (k == 0 || q < Q[j]) ? q : Q[j];
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < CH; ++j)
                if ((AT > 0 || c0 + j < A) && Q[j] > best_q) { best_q = Q[j]; best_idx = base + c0 + j; }  // strict: first minimum of J
        }
    };
    if (h == 1) {
        if (tid == 0) leaves(0.0, 0.0, prev_q, 0, [&](int, double& rt, double& b) { rt = 0.0; b = buf0; });
        SearchOut o; o.q = best_q; o.idx = best_idx;
        return o;
    }
    double thresh = __longlong_as_double(0xfff0000000000000ll);
    for (int p0 = 0; p0 < n_prefix; p0 += nthreads) {   // uniform trip count: the warp shares its best value per round
        if (PRUNE) {
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
        int dig[kScenMaxH];
        int rem = p;
#pragma unroll
        for (int i = kScenMaxH - 3; i >= 0; --i) {
            if (i < P) { dig[i] = rem % A; rem /= A; }
        }
        // the prefix's state per scenario into the scratch; vq, qv and the last action are the same for every scenario
        double vq = 0.0, qv = 0.0;
        int ap = prev_q;
        for (int k = 0; k < K; ++k) {
            double vqk = 0.0, qvk = 0.0, rt = 0.0, b = buf0;
            int apk = prev_q;
#pragma unroll
            for (int i = 0; i < kScenMaxH - 2; ++i) {
                if (i < P) {
                    const int a = dig[i];
                    const double u = sU[i * A + a];
                    const double up = apk >= 0 ? sU[i * A + apk] : u;
                    const double rb = sRB[(k * H + i) * A + a];
                    interior<true>(vqk, qvk, rt, b, u, fabs(dsub(u, up)), rb, rb, L, B);
                    apk = a;
                }
            }
            ps[(2 * k) * kScenThreads] = rt;
            ps[(2 * k + 1) * kScenThreads] = b;
            vq = vqk; qv = qvk; ap = apk;
        }
        if (PRUNE && ap >= 0) {   // bound over the last two levels
            if (scen_bound<OBJ>(vq, qv, [&](int k) { return ps[(2 * k) * kScenThreads]; }, K, sW, g45[ap], vw, rw) < thresh)
                continue;
        }
        const double up4 = ap >= 0 ? sU[i4 * A + ap] : 0.0;
#pragma unroll 1
        for (int a4 = 0; a4 < A; ++a4) {
            const double u4 = sU[i4 * A + a4];
            const double du4 = ap >= 0 ? fabs(dsub(u4, up4)) : 0.0;
            const double vq4 = dadd(vq, u4), qv4 = dadd(qv, du4);
            auto child = [&](const int k, double& rt, double& b) {
                double x = vq, y = qv;
                rt = ps[(2 * k) * kScenThreads];
                b = ps[(2 * k + 1) * kScenThreads];
                const double rb = sRB[(k * H + i4) * A + a4];
                interior<true>(x, y, rt, b, u4, du4, rb, rb, L, B);
            };
            if (PRUNE) {   // bound over the last level
                const double t4 = best_q > thresh ? best_q : thresh;
                auto rt_of = [&](const int k) { double rt, b; child(k, rt, b); return rt; };
                if (scen_bound<OBJ>(vq4, qv4, rt_of, K, sW, g5[a4], vw, rw) < t4) continue;
            }
            leaves(vq4, qv4, a4, (p * A + a4) * A, child);
        }
    }
    SearchOut o; o.q = best_q; o.idx = best_idx;
    return o;
}

// WPS warps per session (the rule of launch_mpc), AT compiled ladder size (0 = runtime A), OBJ ABR_MPC_SCEN_MEAN or
// ABR_MPC_SCEN_WORST, PRUNE branch and bound (both penalties >= 0, no ABR_MPC_EXHAUSTIVE).  K is a runtime value: the
// tables and the threads' scratch are sized by the call in dynamic shared memory.
template <int WPS, int AT, int OBJ, bool PRUNE>
__global__ void __launch_bounds__(kScenThreads) abr_mpc_scen_kernel(const MpcScenArgs a) {
    extern __shared__ double scen_smem[];
    constexpr int SPB = kScenWarpsPerBlock / WPS;
    constexpr int NT = 32 * WPS;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int slot = warp / WPS, wis = warp % WPS, tid = wis * 32 + lane;
    const AbrParams& p = a.p;
    const int A = AT > 0 ? AT : a.A, H = a.H, K = a.K;
    const double L = p.chunk_length, B = p.max_buffer, vw = p.smooth_penalty, rw = p.rebuf_penalty;
    const double inf = __longlong_as_double(0x7ff0000000000000ll);
    double* sU = scen_smem + slot * scen_slot_doubles(A, H, K);
    double* sRB = sU + H * A;
    double* sAD = sRB + K * H * A;
    double* sW = sAD + A * A;
    double* g5 = sW + K;
    double* g45 = g5 + A;
    double* redq = g45 + A;
    int* redi = reinterpret_cast<int*>(redq + kScenWarpsPerBlock);
    double* ps = scen_smem + SPB * scen_slot_doubles(A, H, K) + threadIdx.x;
    auto barrier = [] { if (WPS > 1) __syncthreads(); else __syncwarp(); };

    for (long long s = (long long)blockIdx.x * SPB + slot; s < a.N; s += (long long)gridDim.x * SPB) {
        // every thread of a session computes the status redundantly and identically (every warp reads every input),
        // so control flow and every barrier are uniform across the session
        const int k0 = a.chunk_idx[s];
        const int prev_q = a.prev_q[s];
        const double buf0 = a.buffer[s];
        int h = H, status = 0, act = -1;   // status: 0 search, 1 fixed action (act), 2 input error
        if (a.done && a.done[s]) { status = 1; act = 0; }
        else if (k0 < 0 || prev_q >= A) status = 2;
        else {
            if (k0 + H > a.V) h = a.V - k0;
            if (h <= 0) { status = 1; act = 0; }
        }
        if (status == 0) {
            bool bad = false;
            for (int e0 = 0; e0 < K * h; e0 += 32) {
                const int e = e0 + lane;
                double x = 1.0;
                if (e < K * h) { const int kk = e / h; x = a.pred[(s * K + kk) * H + (e - kk * h)]; }
                bad |= __ballot_sync(0xffffffffu, !(x > 0.0 && x < inf)) != 0u;
            }
            if (OBJ == ABR_MPC_SCEN_MEAN && a.weight) {   // K <= 16: one lane per weight
                const double x = lane < K ? a.weight[s * K + lane] : 0.0;
                bad |= __ballot_sync(0xffffffffu, !(x >= 0.0 && x < inf)) != 0u;
                bad |= __ballot_sync(0xffffffffu, x > 0.0) == 0u;
            }
            if (bad) status = 2;
            else {
                for (int e = tid; e < K * h * A; e += NT) {
                    const int kk = e / (h * A), r = e - kk * (h * A), i = r / A, aa = r - i * A;
                    ABR_CHECK(k0 + i < a.V, "scenario table entry");
                    sRB[(kk * H + i) * A + aa] = ddiv(a.sizes[(k0 + i) * A + aa], a.pred[(s * K + kk) * H + i]);
                }
                for (int e = tid; e < h * A; e += NT) sU[e] = a.util[k0 * A + e];
                if (OBJ == ABR_MPC_SCEN_MEAN)
                    for (int kk = tid; kk < K; kk += NT) sW[kk] = a.weight ? a.weight[s * K + kk] : ddiv(1.0, (double)K);
            }
        }
        barrier();
        SearchOut o; o.q = 0.0; o.idx = 0;
        if (status == 0) {
            const int i5 = h - 1;
            for (int e = tid; e < A * A; e += NT) {
                const int a5 = e / A, a4 = e - a5 * A;
                sAD[e] = fabs(dsub(sU[i5 * A + a5], sU[i5 * A + a4]));
            }
            if (PRUNE && h >= 2) bound_tables(sU, A, h, vw, g5, g45, lane);
            barrier();
            o = scen_search<AT, OBJ, PRUNE>(sU, sRB, sAD, sW, g5, g45, ps, A, H, K, h, prev_q, buf0, vw, rw, L, B, tid, NT);
            // ---- argmin over the session's threads: key (J, linear index) ----
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                const double oq = __shfl_xor_sync(0xffffffffu, o.q, off);
                const int oi = __shfl_xor_sync(0xffffffffu, o.idx, off);
                better(o.q, o.idx, oq, oi);
            }
            if (WPS > 1) {
                if (lane == 0) { redq[wis] = o.q; redi[wis] = o.idx; }
                __syncthreads();
                o.q = redq[0]; o.idx = redi[0];
                for (int w = 1; w < WPS; ++w) better(o.q, o.idx, redq[w], redi[w]);
            }
        }
        if (tid == 0) {
            if (status == 0) {
                const int idx = o.idx == 0x7fffffff ? 0 : o.idx;   // all aggregates -inf/NaN: first sequence
                int div = 1, first = idx;
                for (int i = 1; i < h; ++i) { div *= A; first /= A; }
                a.action[s] = first;
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
                if (a.best_j) a.best_j[s] = __longlong_as_double(0x7ff8000000000000ll);
                if (a.best_seq) for (int i = 0; i < H; ++i) a.best_seq[s * H + i] = -1;
                if (status == 2 && a.error_count64) atomicAdd(a.error_count64, 1ull);
            }
        }
        barrier();   // tables and the reduction slots are reused by the next session of this slot
    }
}

}  // namespace

template <int WPS, int AT, int OBJ, bool PRUNE>
static cudaError_t run_mpc_scen(const MpcScenArgs& a, const unsigned grid, const size_t smem, cudaStream_t st) {
    if (smem > 48 * 1024) {   // past the default limit of dynamic shared memory (K = 16 with the larger shapes)
        const cudaError_t e = cudaFuncSetAttribute(abr_mpc_scen_kernel<WPS, AT, OBJ, PRUNE>,
                                                   cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    abr_mpc_scen_kernel<WPS, AT, OBJ, PRUNE><<<grid, kScenThreads, smem, st>>>(a);
    return cudaSuccess;
}

template <int WPS, int AT>
static cudaError_t run_mpc_scen_obj(const MpcScenArgs& a, const bool prune, const unsigned grid, const size_t smem,
                                    cudaStream_t st) {
    if (a.objective == ABR_MPC_SCEN_WORST)
        return prune ? run_mpc_scen<WPS, AT, ABR_MPC_SCEN_WORST, true>(a, grid, smem, st)
                     : run_mpc_scen<WPS, AT, ABR_MPC_SCEN_WORST, false>(a, grid, smem, st);
    return prune ? run_mpc_scen<WPS, AT, ABR_MPC_SCEN_MEAN, true>(a, grid, smem, st)
                 : run_mpc_scen<WPS, AT, ABR_MPC_SCEN_MEAN, false>(a, grid, smem, st);
}

template <int AT>
static cudaError_t run_mpc_scen_wps(const MpcScenArgs& a, const int wps, const bool prune, const unsigned grid,
                                    const size_t smem, cudaStream_t st) {
    return wps == 1 ? run_mpc_scen_obj<1, AT>(a, prune, grid, smem, st)
                    : run_mpc_scen_obj<kScenWarpsPerBlock, AT>(a, prune, grid, smem, st);
}

cudaError_t launch_mpc_scen(const MpcScenArgs& a, cudaStream_t st) {
    if (a.N <= 0) return cudaSuccess;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    // warps per session and grid: the rule of launch_mpc
    long long combos = 1;
    for (int i = 0; i < a.H; ++i) combos *= a.A;
    const int wps = (a.N >= (long long)sms * 16 || combos < 32 * 36 * 4) ? 1 : kScenWarpsPerBlock;
    const int spb = kScenWarpsPerBlock / wps;
    long long blocks = (a.N + spb - 1) / spb;
    if (blocks > (long long)sms * 64) blocks = (long long)sms * 64;
    const bool prune = !(a.flags & ABR_MPC_EXHAUSTIVE) && a.p.smooth_penalty >= 0.0 && a.p.rebuf_penalty >= 0.0;
    const size_t smem = (size_t)(spb * scen_slot_doubles(a.A, a.H, a.K) + 2 * a.K * kScenThreads) * sizeof(double);
    const unsigned g = (unsigned)blocks;
    cudaError_t e;
    switch (a.A) {
        case 2: e = run_mpc_scen_wps<2>(a, wps, prune, g, smem, st); break;
        case 3: e = run_mpc_scen_wps<3>(a, wps, prune, g, smem, st); break;
        case 4: e = run_mpc_scen_wps<4>(a, wps, prune, g, smem, st); break;
        case 5: e = run_mpc_scen_wps<5>(a, wps, prune, g, smem, st); break;
        case 6: e = run_mpc_scen_wps<6>(a, wps, prune, g, smem, st); break;
        case 8: e = run_mpc_scen_wps<8>(a, wps, prune, g, smem, st); break;
        default: e = run_mpc_scen_wps<0>(a, wps, prune, g, smem, st); break;
    }
    if (e != cudaSuccess) return e;
    count_launch();
    return cudaGetLastError();
}

}  // namespace abr
