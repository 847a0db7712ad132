// Session order by trace (DESIGN.md §4): sessions are independent (Simulator.py:93-131 holds exactly one), so the
// order in which an environment keeps them is free.  Kept sorted by trace, every thread block of the step kernels
// follows one trace and takes the shared-memory path whatever order the caller's sessions come in.
//
// abr_sort_by_trace builds that order: perm[p] = caller's index of the session at environment position p, a stable
// (hence deterministic) radix sort of (trace id, session index) pairs, an invalid trace id (< 0 or >= n_traces) keyed
// as trace 0, the trace the reset puts such a session on.  Set-up code, run once per session->trace assignment; the
// radix sort itself is CUB's (header-only, part of the CUDA toolkit).
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "abr_common.cuh"

namespace abr {

namespace {

// The radix sort's pairs: the trace id as the counting sort buckets it (an invalid id as trace 0; the raw id would
// sort by its low end_bit bits, -1 after every trace) and the session index.
__global__ void __launch_bounds__(256)
abr_sort_keys_kernel(const int32_t* __restrict__ tid, int n, int n_traces, int32_t* __restrict__ keys, int32_t* __restrict__ iota) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int t = tid[i];
    keys[i] = (t < 0 || t >= n_traces) ? 0 : t;
    iota[i] = i;
}

// ---- counting sort by trace, fused with the gather of the reset's inputs (abr_env_reset_sorted) ----
// The sessions are cut into n_blocks runs of S consecutive sessions.  hist[trace][block] first counts the sessions
// of each trace in each run, an exclusive scan in that (trace-major) order turns the counts into the first output
// position of every (trace, run), and one warp per run then walks its sessions in order and places them: stable,
// hence deterministic — the same order as the radix sort above, invalid ids included.  Three small launches instead
// of CUB's sort, its key pass, a copy of the order and two gathers.

__global__ void __launch_bounds__(256)
abr_sort_count(const int32_t* __restrict__ tid, int n, int S, int n_traces, int n_blocks, int32_t* __restrict__ hist) {
    const int b = blockIdx.x;
    const int hi = min(n, (b + 1) * S);
    for (int i = b * S + threadIdx.x; i < hi; i += blockDim.x) {
        const int t = tid[i];
        const int bucket = (t < 0 || t >= n_traces) ? 0 : t;      // an invalid id is flagged by the reset; it sorts as trace 0
        atomicAdd(hist + (size_t)bucket * n_blocks + b, 1);
    }
}

// One block per run of S sessions (a multiple of kSortChunk); the run's cursors (first free position per trace) live
// in shared memory.  The block takes kSortChunk sessions at a time: all threads fetch the trace ids, warp 0 ranks them
// in order — rounds of 32 consecutive sessions, the serial part of a round being a handful of ballots and one
// shared-memory atomic — and all threads then scatter the sessions to their positions (every one of those stores is a
// sector of its own in the interleaved layout: they want as many warps as possible).
constexpr int kSortChunk = 512;
constexpr int kSortThreads = 256;

__global__ void __launch_bounds__(kSortThreads)
abr_sort_place(const int32_t* __restrict__ tid, const double* __restrict__ off, int n, int S, int n_traces, int n_blocks,
               int key_bits, int32_t* __restrict__ hist, int32_t* __restrict__ perm, int32_t* __restrict__ tid_sorted,
               double* __restrict__ off_sorted) {
    extern __shared__ int s_dyn[];
    int* s_tid = s_dyn;                   // [kSortChunk]
    int* s_pos = s_dyn + kSortChunk;      // [kSortChunk]
    int* s_cur = s_dyn + 2 * kSortChunk;  // [n_traces]
    const int b = blockIdx.x, x = threadIdx.x, lane = x & 31;
    // the run's cursors (the cells are n_blocks apart: every load is its own sector; four in flight per thread);
    // the cells are left at zero for the next call's counting pass (no memset in front of it)
    for (int t0 = x; t0 < n_traces; t0 += kSortThreads * 4) {
        int c[4];
#pragma unroll
        for (int k = 0; k < 4; ++k)
            c[k] = t0 + kSortThreads * k < n_traces ? __ldcg(hist + (size_t)(t0 + kSortThreads * k) * n_blocks + b) : 0;
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (t0 + kSortThreads * k < n_traces) {
                s_cur[t0 + kSortThreads * k] = c[k];
                hist[(size_t)(t0 + kSortThreads * k) * n_blocks + b] = 0;
            }
    }
    const int hi = min(n, (b + 1) * S);
    for (int c0 = b * S; c0 < hi; c0 += kSortChunk) {
#pragma unroll
        for (int j = x; j < kSortChunk; j += kSortThreads) s_tid[j] = c0 + j < hi ? tid[c0 + j] : -1;
        __syncthreads();                   // trace ids (and, the first time, the cursors) are in place
        if (x < 32) {
#pragma unroll 4
            for (int k = 0; k < kSortChunk / 32; ++k) {
                const bool valid = c0 + 32 * k + lane < hi;
                const int t = s_tid[32 * k + lane];
                const int bucket = (t < 0 || t >= n_traces) ? 0 : t;
                // Lanes of the same trace take consecutive positions in lane order.  The lanes that share this lane's
                // trace, from one ballot per key bit (a match.any instruction walks the distinct keys one by one: 32 of
                // them in the interleaved layout); idle lanes of the last round are masked out.
                unsigned peers = __ballot_sync(0xffffffffu, valid);
                for (int bit = 0; bit < key_bits; ++bit) {
                    const bool one = (bucket >> bit) & 1;
                    const unsigned vote = __ballot_sync(0xffffffffu, one);
                    peers &= one ? vote : ~vote;
                }
                const int rank = __popc(peers & ((1u << lane) - 1u));
                // the group's first lane takes the group's positions from the trace's cursor (a shared-memory atomic:
                // the rounds need no barrier between them, the cursor's updates stay in program order) and hands the
                // first one to the others
                const int leader = valid ? __ffs(peers) - 1 : lane;
                int base = 0;
                ABR_CHECK(bucket >= 0 && bucket < n_traces && (!valid || (peers >> lane) & 1u), "trace cursor / peer group");
                if (valid && lane == leader) base = atomicAdd(&s_cur[bucket], __popc(peers));
                base = __shfl_sync(0xffffffffu, base, leader);
                s_pos[32 * k + lane] = base + rank;
            }
        }
        __syncthreads();
#pragma unroll
        for (int j = x; j < kSortChunk; j += kSortThreads) {
            const int i = c0 + j;
            if (i < hi) {
                const int pos = s_pos[j];
                ABR_CHECK(pos >= 0 && pos < n, "position of a session in the sorted order");
                perm[pos] = i;
                tid_sorted[pos] = s_tid[j];
                off_sorted[pos] = off ? off[i] : 0.0;
            }
        }
        __syncthreads();                   // s_tid / s_pos are rewritten by the next chunk
    }
}

__global__ void __launch_bounds__(256)
abr_gather_kernel(const int32_t* __restrict__ tid, const double* __restrict__ off, const int32_t* __restrict__ perm, int n,
                  int32_t* __restrict__ tid_sorted, double* __restrict__ off_sorted) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const int i = perm[p];
    tid_sorted[p] = tid[i];
    off_sorted[p] = off ? off[i] : 0.0;
}

}  // namespace

cudaError_t launch_gather(const int32_t* d_trace_id, const double* d_off, const int32_t* d_perm, int n,
                          int32_t* d_tid_sorted, double* d_off_sorted, cudaStream_t st) {
    abr_gather_kernel<<<(n + 255) / 256, 256, 0, st>>>(d_trace_id, d_off, d_perm, n, d_tid_sorted, d_off_sorted);
    count_launch();
    return cudaGetLastError();
}

// Shape of the counting sort for n sessions over n_traces traces: runs of S sessions, n_blocks of them; 0 blocks when
// the shape does not fit (cursor table beyond 48 KB of shared memory, or too many (trace, run) cells for a one-block scan).
void sort_shape(int n, int n_traces, int* S, int* n_blocks) {
    *S = kSortChunk; *n_blocks = 0;
    if (n <= 0 || n_traces > 11264) return;          // cursors + the chunk's buffers within 48 KB of shared memory
    long long blocks = ((long long)n + *S - 1) / *S;
    const long long max_cells = 1 << 18;
    while (blocks * n_traces > max_cells && *S < (1 << 20)) { *S *= 2; blocks = ((long long)n + *S - 1) / *S; }
    if (blocks * n_traces > max_cells) return;
    *n_blocks = (int)blocks;
}

// bytes of scratch behind the cells that the scan needs
size_t sort_scan_tmp_bytes(int total) {
    size_t bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, bytes, (int32_t*)nullptr, (int32_t*)nullptr, total);
    return (bytes + 255) & ~(size_t)255;
}

// d_hist: n_traces * n_blocks ints of scratch (sort_shape), all zero on entry and left all zero; d_scan_tmp: scratch
// of sort_scan_tmp_bytes.  Outputs: the order, and the trace ids / start offsets
// gathered into that order (what abr_env_reset then reads).
cudaError_t launch_sort_gather(const int32_t* d_trace_id, const double* d_off, int n, int n_traces, int S, int n_blocks,
                               int32_t* d_hist, void* d_scan_tmp, size_t scan_tmp_bytes, int32_t* d_perm,
                               int32_t* d_tid_sorted, double* d_off_sorted, cudaStream_t st) {
    const int total = n_traces * n_blocks;
    int key_bits = 0;
    while ((1 << key_bits) < n_traces) ++key_bits;
    abr_sort_count<<<n_blocks, 256, 0, st>>>(d_trace_id, n, S, n_traces, n_blocks, d_hist);
    // exclusive scan of the cells in place (CUB's decoupled look-back scan: an init kernel and the scan)
    cudaError_t e = cub::DeviceScan::ExclusiveSum(d_scan_tmp, scan_tmp_bytes, d_hist, d_hist, total, st);
    if (e != cudaSuccess) return e;
    abr_sort_place<<<n_blocks, kSortThreads, sizeof(int) * ((size_t)n_traces + 2 * kSortChunk), st>>>(d_trace_id, d_off, n, S, n_traces, n_blocks, key_bits,
                                                                        d_hist, d_perm, d_tid_sorted, d_off_sorted);
    count_launch(4);
    return cudaGetLastError();
}

// d_tmp: caller-provided scratch of *tmp_bytes bytes; with d_tmp == nullptr only *tmp_bytes is set (layout:
// [keys n][sorted keys n][iota n][CUB temp storage]).
cudaError_t launch_sort_by_trace(const int32_t* d_trace_id, int n, int n_traces, int32_t* d_perm, void* d_tmp,
                                 size_t* tmp_bytes, cudaStream_t st) {
    int end_bit = 1;
    while (end_bit < 31 && (1ll << end_bit) < (long long)n_traces) ++end_bit;
    size_t cub_bytes = 0;
    cudaError_t e = cub::DeviceRadixSort::SortPairs(nullptr, cub_bytes, (const int32_t*)nullptr, (int32_t*)nullptr,
                                                    (const int32_t*)nullptr, (int32_t*)nullptr, n, 0, end_bit, st);
    if (e != cudaSuccess) return e;
    const size_t arr = ((size_t)n * sizeof(int32_t) + 255) & ~(size_t)255;
    if (!d_tmp) { *tmp_bytes = 3 * arr + cub_bytes; return cudaSuccess; }
    int32_t* keys_in = reinterpret_cast<int32_t*>(d_tmp);
    int32_t* keys_out = reinterpret_cast<int32_t*>(reinterpret_cast<char*>(d_tmp) + arr);
    int32_t* iota = reinterpret_cast<int32_t*>(reinterpret_cast<char*>(d_tmp) + 2 * arr);
    void* cub_tmp = reinterpret_cast<char*>(d_tmp) + 3 * arr;
    abr_sort_keys_kernel<<<(n + 255) / 256, 256, 0, st>>>(d_trace_id, n, n_traces, keys_in, iota);
    count_launch();
    e = cub::DeviceRadixSort::SortPairs(cub_tmp, cub_bytes, keys_in, keys_out, iota, d_perm, n, 0, end_bit, st);
    count_launch(2);
    return e != cudaSuccess ? e : cudaGetLastError();
}

}  // namespace abr
