// Matched cosine similarity of synergy sets, fp64: the standard comparison of two sets of synergies of the same rank.
//
// For a pair (a, b) of sets (k x m, row-major, 1 <= k <= 16, 1 <= m <= 64):
//   S[i][j] = <a_i, b_j> / (||a_i|| ||b_j||), 0 where either row has norm 0 (NaN never enters the matching);
//   an exact maximum-weight perfect matching on S - what scipy.optimize.linear_sum_assignment(S, maximize=True)
//   finds - by the O(k^3) shortest augmenting path method (Jonker-Volgenant without initialisation, the variant scipy
//   implements): rows are added one at a time, each by a Dijkstra search over reduced costs of C = -S, with row duals
//   u and column duals v updated after each search;
//   mean[p] = the mean matched similarity; perm[p][i] = the row of b paired with row i of a; sim[p][i] = S[i][perm[i]].
//
// Tie rule: where several unvisited columns share the smallest tentative distance of a search step, the lowest column
// index is taken (scipy prefers a column that is still free, then its own scan order).  Both reach the same optimum;
// where the optimum is not unique the pairings may differ, never the total.
//
// Thread mapping: a tile of G = the next power of two >= max(kmax, 2) lanes owns a pair (256 / G pairs per
// 256-thread CTA, grid-stride over the pairs; a one-lane tile spilled).  Lane j computes column j of S (the rows of a are warp-broadcast loads, row j of b is the
// lane's own stream) and holds column j's dual, tentative distance, predecessor row and assignment; lane i also holds
// row i's dual and assignment.  C = -S of the pair sits in shared memory (G x G doubles).  A search step is: every
// unvisited column relaxes against the current row, a shuffle min-reduction over the tile finds the smallest distance,
// a ballot picks its lowest column.  The norms are computed once per set by ms_sm_norm_kernel, not once per pair.
//
// No floating-point atomics; the tile's sum of the matched similarities is a fixed butterfly: repeated calls are
// bit-identical.  Registers: see DESIGN.md section 7 (-Xptxas -v; no local memory).
#include <stdio.h>

#include <cooperative_groups.h>

#include "ms_common.cuh"

namespace cg = cooperative_groups;

#define SM_MAX_K 16
#define SM_MAX_M 64
#define SM_THREADS 256
#define SM_MAX_CTAS (1 << 16)
#define SM_BAD_SET 1u
#define SM_BAD_PAIR 2u

// workspace: [0, 256) status word (SM_BAD_*), then 1 / ||row|| (0 for a zero row) of row i of set s at [s * 16 + i]
static inline size_t sm_norms_offset() { return 256; }

__global__ void __launch_bounds__(SM_THREADS) ms_sm_norm_kernel(const double* __restrict__ H, int m,
                                                                const ms_synergy_set* __restrict__ sets, int n_sets,
                                                                int kmax, double* __restrict__ rnorm,
                                                                unsigned* __restrict__ status) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (long long)n_sets * SM_MAX_K) return;
    const int s = (int)(t / SM_MAX_K), i = (int)(t % SM_MAX_K);
    const ms_synergy_set st = sets[s];
    if (st.k < 1 || st.k > kmax || st.offset < 0) {
        if (i == 0) atomicOr(status, SM_BAD_SET);
        return;
    }
    if (i >= st.k) return;
    const double* row = H + st.offset + (long long)i * m;
    double ss = 0.0;
    for (int j = 0; j < m; j++) ss = fma(row[j], row[j], ss);
    const double nrm = sqrt(ss);
    // a zero row has similarity 0 with everything (one whose squared norm overflows too: its norm is inf)
    rnorm[t] = nrm > 0.0 && nrm < INFINITY ? 1.0 / nrm : 0.0;
}

// Pair p of every pair a < b of n sets, in np.triu_indices(n, 1) order, counted from the end: q = P - 1 - p lies in
// the block of row a = n - 2 - r, r = the largest with r (r + 1) / 2 <= q (a block of r + 1 pairs), and b = n - 1 -
// (q - r (r + 1) / 2).  A single-precision square root only seeds r; the integer steps make it exact.
__device__ __forceinline__ int2 sm_triu_pair(long long p, int n) {
    const long long q = (long long)n * (n - 1) / 2 - 1 - p;
    const float x = 8.0f * (float)q + 1.0f;
    long long r = (long long)((x * rsqrtf(x) - 1.0f) * 0.5f);
    while ((r + 1) * (r + 2) / 2 <= q) r++;
    while (r * (r + 1) / 2 > q) r--;
    return make_int2((int)(n - 2 - r), (int)(n - 1 - (q - r * (r + 1) / 2)));
}

// 4 CTAs (32 warps) per SM, 64 registers: without the minimum, ptxas held the G = 4 tile to 48 registers and spilled
template <int G>
__global__ void __launch_bounds__(SM_THREADS, 4) ms_sm_match_kernel(const double* __restrict__ H, int m,
                                                                 const ms_synergy_set* __restrict__ sets, int n_sets,
                                                                 int kmax, const int2* __restrict__ pairs,
                                                                 long long n_pairs, const double* __restrict__ rnorm,
                                                                 int8_t* __restrict__ perm, double* __restrict__ sim,
                                                                 double* __restrict__ mean, unsigned* __restrict__ status) {
    constexpr int GROUPS = SM_THREADS / G;
    __shared__ double sC[GROUPS][G * G];  // C = -S of the tile's pair, row-major
    const cg::thread_block_tile<G> tile = cg::tiled_partition<G>(cg::this_thread_block());
    const int lane = (int)tile.thread_rank();
    double* C = sC[threadIdx.x / G];
    const long long stride = (long long)gridDim.x * GROUPS;
    for (long long p = (long long)blockIdx.x * GROUPS + threadIdx.x / G; p < n_pairs; p += stride) {
        const int2 ab = pairs ? pairs[p] : sm_triu_pair(p, n_sets);
        bool ok = ab.x >= 0 && ab.x < n_sets && ab.y >= 0 && ab.y < n_sets;
        ms_synergy_set sa = {0, 0, 0}, sb = {0, 0, 0};
        if (ok) {
            sa = sets[ab.x];
            sb = sets[ab.y];
            ok = sa.k == sb.k && sa.k >= 1 && sa.k <= kmax && sa.offset >= 0 && sb.offset >= 0;
        }
        if (!ok) {  // tile-uniform: every lane read the same pair
            if (lane == 0) {
                atomicOr(status, SM_BAD_PAIR);
                mean[p] = __longlong_as_double(0x7ff8000000000000ll);
            }
            for (int i = lane; i < kmax; i += G) {
                if (perm) perm[p * kmax + i] = -1;
                if (sim) sim[p * kmax + i] = __longlong_as_double(0x7ff8000000000000ll);
            }
            continue;
        }
        const int k = sa.k;
        const bool col = lane < k;

        // column `lane` of S, stored negated: C[i][lane] = -<a_i, b_lane / ||b_lane||> / ||a_i||.  Every entry of C is
        // finite, which the searches below need to end: b_lane is scaled to unit length as it is loaded, so for a row
        // a_i whose squared norm is finite |acc[i]| <= ||a_i|| cannot overflow, and a row with ra or rb 0 (norm 0, or
        // one that overflows) gets 0 without its sum being looked at.
        if (col) {
            double acc[G];
#pragma unroll
            for (int i = 0; i < G; i++) acc[i] = 0.0;
            const double* A = H + sa.offset;
            const double* B = H + sb.offset + (long long)lane * m;
            const double rb = rnorm[(long long)ab.y * SM_MAX_K + lane];
            for (int t = 0; t < m; t++) {
                const double bj = __ldg(B + t) * rb;
#pragma unroll
                for (int i = 0; i < G; i++)
                    if (i < k) acc[i] = fma(__ldg(A + i * m + t), bj, acc[i]);
            }
            const double* ra = rnorm + (long long)ab.x * SM_MAX_K;
#pragma unroll
            for (int i = 0; i < G; i++)
                if (i < k) C[i * G + lane] = ra[i] == 0.0 || rb == 0.0 ? 0.0 : -(acc[i] * ra[i]);
        }
        tile.sync();

        // shortest augmenting paths (scipy's rectangular_lsap, square case), one row added per search
        double v = 0.0, u = 0.0;  // dual of column `lane`, dual of row `lane`
        int row4col = -1, col4row = -1;
        for (int cur = 0; cur < k; cur++) {
            double spc = INFINITY, min_val = 0.0;  // tentative distance of column `lane`, distance reached
            int path = -1, i = cur, sink = cur;
            bool sc = !col, sr = false;  // column `lane` visited (or absent), row `lane` visited
            // each step visits a new column, so with a finite C a free one is reached within k steps; the bound only
            // guarantees that the tile never loops
            for (int step = 0; step < k; step++) {
                sr |= lane == i;
                const double ui = tile.shfl(u, i);
                if (!sc) {
                    const double r = min_val + C[i * G + lane] - ui - v;
                    if (r < spc) {
                        spc = r;
                        path = i;
                    }
                }
                const double cand = sc ? INFINITY : spc;
                double low = cand;
#pragma unroll
                for (int off = G / 2; off > 0; off >>= 1) low = fmin(low, tile.shfl_xor(low, off));
                const int j = __ffs(tile.ballot(cand == low)) - 1;  // tie rule: lowest column
                min_val = low;
                const int r4c = tile.shfl(row4col, j);
                sc |= lane == j;
                if (r4c < 0) {
                    sink = j;
                    break;
                }
                i = r4c;
            }
            const double spc_own = tile.shfl(spc, col4row < 0 ? 0 : col4row);  // distance of this row's column
            if (lane == cur)
                u += min_val;
            else if (sr)
                u += min_val - spc_own;
            if (col && sc) v -= min_val - spc;
            for (int j = sink, step = 0; step < k; step++) {  // augment along the predecessors back to row `cur`
                const int r = tile.shfl(path, j);
                if (lane == j) row4col = r;
                const int prev = tile.shfl(col4row, r);
                if (lane == r) col4row = j;
                j = prev;
                if (r == cur) break;
            }
        }

        const double s = col ? -C[lane * G + col4row] : 0.0;
        double total = s;
#pragma unroll
        for (int off = G / 2; off > 0; off >>= 1) total += tile.shfl_xor(total, off);  // same sum in every lane
        if (lane == 0) mean[p] = total / k;
        for (int i = lane; i < kmax; i += G) {
            if (perm) perm[p * kmax + i] = (int8_t)(i < k ? col4row : -1);
            if (sim) sim[p * kmax + i] = i < k ? s : __longlong_as_double(0x7ff8000000000000ll);
        }
        tile.sync();  // C is rewritten by the next pair
    }
}

extern "C" int64_t ms_synergy_match_workspace_bytes(int32_t n_sets) {
    if (n_sets < 0) return 0;
    return (int64_t)sm_norms_offset() + (int64_t)n_sets * SM_MAX_K * (int64_t)sizeof(double);
}

template <int G>
static void sm_launch(const double* d_H, int32_t m, const ms_synergy_set* d_sets, int32_t n_sets, int32_t kmax,
                      const int32_t* d_pairs, int64_t n_pairs, int8_t* d_perm, double* d_sim, double* d_mean,
                      const double* rnorm, unsigned* status, cudaStream_t st) {
    constexpr int GROUPS = SM_THREADS / G;
    const long long need = (n_pairs + GROUPS - 1) / GROUPS;
    const int ctas = (int)(need < SM_MAX_CTAS ? need : SM_MAX_CTAS);
    ms_sm_match_kernel<G><<<ctas, SM_THREADS, 0, st>>>(d_H, m, d_sets, n_sets, kmax, (const int2*)d_pairs, n_pairs,
                                                       rnorm, d_perm, d_sim, d_mean, status);
}

extern "C" int ms_synergy_match(const double* d_H, int32_t m, const ms_synergy_set* d_sets, int32_t n_sets,
                                int32_t kmax, const int32_t* d_pairs, int64_t n_pairs, int8_t* d_perm, double* d_sim,
                                double* d_mean, void* d_work, int64_t work_bytes, void* stream) {
    if (m < 1 || m > SM_MAX_M || kmax < 1 || kmax > SM_MAX_K || n_sets < 0 || n_pairs < 0) return MS_E_INVALID;
    if (n_pairs == 0) return MS_OK;
    if (!d_H || !d_sets || !d_mean || !d_work || n_sets == 0) return MS_E_INVALID;
    if (!d_pairs && n_pairs != (int64_t)n_sets * (n_sets - 1) / 2) return MS_E_INVALID;  // NULL: every pair a < b
    if (((uintptr_t)d_pairs & 7) != 0 || ((uintptr_t)d_work & 7) != 0) return MS_E_INVALID;
    if (work_bytes < ms_synergy_match_workspace_bytes(n_sets)) return MS_E_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    unsigned* status = (unsigned*)d_work;
    double* rnorm = (double*)((char*)d_work + sm_norms_offset());
    MS_CUDA_CHECK(cudaMemsetAsync(status, 0, sizeof(unsigned), st));
    const long long rows = (long long)n_sets * SM_MAX_K;
    ms_sm_norm_kernel<<<(unsigned)((rows + SM_THREADS - 1) / SM_THREADS), SM_THREADS, 0, st>>>(d_H, m, d_sets, n_sets,
                                                                                             kmax, rnorm, status);
    MS_COUNT_LAUNCH();
    if (kmax <= 2)
        sm_launch<2>(d_H, m, d_sets, n_sets, kmax, d_pairs, n_pairs, d_perm, d_sim, d_mean, rnorm, status, st);
    else if (kmax <= 4)
        sm_launch<4>(d_H, m, d_sets, n_sets, kmax, d_pairs, n_pairs, d_perm, d_sim, d_mean, rnorm, status, st);
    else if (kmax <= 8)
        sm_launch<8>(d_H, m, d_sets, n_sets, kmax, d_pairs, n_pairs, d_perm, d_sim, d_mean, rnorm, status, st);
    else
        sm_launch<16>(d_H, m, d_sets, n_sets, kmax, d_pairs, n_pairs, d_perm, d_sim, d_mean, rnorm, status, st);
    MS_COUNT_LAUNCH();
    MS_CUDA_CHECK(cudaGetLastError());
    // the set table and the pair list are device data: their check travels back with the status word
    unsigned h_status = 0;
    MS_CUDA_CHECK(cudaMemcpyAsync(&h_status, status, sizeof(unsigned), cudaMemcpyDeviceToHost, st));
    MS_CUDA_CHECK(cudaStreamSynchronize(st));
    return h_status ? MS_E_INVALID : MS_OK;
}
