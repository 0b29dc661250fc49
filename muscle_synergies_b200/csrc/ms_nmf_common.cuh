// What the four NMF solver families (ms_nmf.cu, ms_nmf_cd.cu, ms_nmf_fixed.cu, ms_nmf_beta.cu) share: the problem table
// and the shapes it supports, the rank dispatch, the fixed-order CTA sum, the shared-memory budget of the resident
// kernels, and the host side of the streaming loops' early stop.
#pragma once
#include <stdio.h>
#include <stdlib.h>

#include "ms_common.cuh"

#define MS_NMF_MAX_K 16  // ranks 1..16, one template instance each
#define MS_NMF_MAX_M 64  // columns (muscles) of X

// The problem table of a batch, 32 bytes per problem (ms_nmf_plan).  Offsets count elements, so the same table serves
// fp32 and fp64 factors.
struct MsNmfProblem {
    int k;
    long long w_off;  // from the packed W to this problem's W [n][k]
    long long h_off;  // from the packed H to this problem's H [k][m]
    long long x_off;  // from X to this problem's X [n][m]
};

// CALL(K) for the compile-time rank K equal to KEXPR; a rank outside 1..16 runs nothing
#define MS_NMF_K_SWITCH(KEXPR, CALL)                                                                                  \
    switch (KEXPR) {                                                                                                  \
        case 1: CALL(1); break;   case 2: CALL(2); break;   case 3: CALL(3); break;   case 4: CALL(4); break;         \
        case 5: CALL(5); break;   case 6: CALL(6); break;   case 7: CALL(7); break;   case 8: CALL(8); break;         \
        case 9: CALL(9); break;   case 10: CALL(10); break; case 11: CALL(11); break; case 12: CALL(12); break;       \
        case 13: CALL(13); break; case 14: CALL(14); break; case 15: CALL(15); break; case 16: CALL(16); break;       \
        default: break;                                                                                               \
    }

__host__ __device__ inline int ms_odd(int v) { return v | 1; }  // row stride in doubles: an odd stride is free of bank conflicts

static inline size_t ms_align256(size_t b) { return (b + 255) / 256 * 256; }

__device__ __forceinline__ double ms_warp_sum_d(double v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// fixed-order sum over the CTA (warp trees, then the warps in order); every thread gets the total.  s_red: one double
// per warp.
__device__ __forceinline__ double ms_block_sum_d(double v, double* s_red) {
    v = ms_warp_sum_d(v);
    __syncthreads();  // s_red is free
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    double total = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) total += s_red[w];
    return total;
}

// Shared memory a resident kernel may take per CTA: 1 KiB below the 227 KiB an sm_100 CTA can have.
static const size_t MS_NMF_SMEM_BUDGET = 227 * 1024 - 1024;

// Largest n for which fixed + n * per_row elements of elem_bytes each fit MS_NMF_SMEM_BUDGET; 0 for a shape outside
// m in 1..64, kmax in 1..16.  fixed(m, kmax) and per_row(m, kmax) are a family's shared-memory layout.
static inline int32_t ms_nmf_max_rows(int32_t m, int32_t kmax, size_t elem_bytes, size_t (*fixed)(int, int),
                                      size_t (*per_row)(int, int)) {
    if (m < 1 || m > MS_NMF_MAX_M || kmax < 1 || kmax > MS_NMF_MAX_K) return 0;
    return (int32_t)((MS_NMF_SMEM_BUDGET - elem_bytes * fixed(m, kmax)) / (elem_bytes * per_row(m, kmax)));
}

// Writes the problem table of a batch to host memory: W_p [n][k_p] and H_p [k_p][m] packed problem after problem, X_p
// the matrix h_x_index[p] (NULL: all 0) of a stack of [n][m] matrices.  Returns the largest rank, or MS_E_INVALID for a
// rank outside 1..16 or a negative matrix index.
static inline int32_t ms_nmf_fill_table(long long n, int m, const int32_t* h_ranks, const int32_t* h_x_index,
                                        int n_problems, MsNmfProblem* h) {
    long long wo = 0, ho = 0;
    int kmax = 0;
    for (int p = 0; p < n_problems; p++) {
        const int k = h_ranks[p];
        if (k < 1 || k > MS_NMF_MAX_K) return MS_E_INVALID;
        h[p].k = k;
        h[p].w_off = wo;
        h[p].h_off = ho;
        h[p].x_off = h_x_index ? (long long)h_x_index[p] * n * m : 0;
        if (h[p].x_off < 0) return MS_E_INVALID;
        wo += n * k;
        ho += (long long)k * m;
        if (k > kmax) kmax = k;
    }
    return kmax;
}

// The early stop of a streaming loop: copies the per-problem states (each with a `done` flag) back - a pageable copy,
// so it waits for the stream - and returns 1 when every problem is done, 0 when one is not, or a negative MS_E_* code.
template <typename State>
static int ms_nmf_all_done(const State* d_states, int n_problems, cudaStream_t st) {
    State* h = (State*)malloc(sizeof(State) * (size_t)n_problems);
    if (!h) return MS_E_INVALID;
    cudaError_t e = cudaMemcpyAsync(h, d_states, sizeof(State) * (size_t)n_problems, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    int all_done = 1;
    for (int p = 0; e == cudaSuccess && p < n_problems; p++) all_done &= h[p].done != 0;
    free(h);
    MS_CUDA_CHECK(e);
    return all_done;
}
