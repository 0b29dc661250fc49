// Batched NMF by coordinate descent (Frobenius loss, fp64) and NNDSVD initialisation - EXTENSION stage.
//
// scikit-learn's default solver, restated for a batch of problems (sklearn 1.9.0,
// sklearn/decomposition/_nmf.py: _fit_coordinate_descent, _update_coordinate_descent; _cdnmf_fast.pyx:
// _update_cdnmf_fast) with shuffle=False and no regularisation.  One iteration:
//
//   W step   HHt = H H^T, XHt = X H^T;  for t = 0..k-1, every row i:
//              grad = -XHt[i,t] + sum_r HHt[t,r] W[i,r]        (W entries already updated in this sweep)
//              violation += |grad| (|min(0, grad)| where W[i,t] == 0)
//              W[i,t] = max(W[i,t] - grad / HHt[t,t], 0)       (when HHt[t,t] != 0)
//   H step   the same on (X^T, H^T, W) with W^T W and X^T W of the UPDATED W
//   stop     violation_init = violation of iteration 1; stop when it is 0 or violation / violation_init <= tol
//
// Rows (W step) and columns of H (H step) are independent, so one thread owns a row and runs its k coordinate steps
// in order: the same arithmetic as sklearn's t-outer / i-inner loop, up to the summation order of the products.
//
//   ms_cd_resident_kernel    one CTA per problem, X / W / H and the Gram matrices in shared memory (fp64)
//   ms_cd_stream_*           long signals: one pass over X and W in HBM per iteration (W step, W^T W, X^T W and the
//                            violation), then one small CTA per problem for the H step and the stop test
//   ms_nndsvd_*              _initialize_nmf(init="nndsvd" / "nndsvda") from an exact SVD: X^T X, cyclic Jacobi,
//                            U = X V S^-1; one SVD per distinct matrix of the stack serves every rank on it
#include <stdio.h>

#include "ms_common.cuh"

#define CD_THREADS 256
#define CD_MAX_K 16
#define CD_MAX_M 64
#define CD_ITEMS ((CD_MAX_K * CD_MAX_K + CD_MAX_K * CD_MAX_M + CD_THREADS - 1) / CD_THREADS)  // reduction items a thread owns

// ms_nmf_plan's table (csrc/ms_nmf.cu): offsets are element counts, so they serve fp64 factors unchanged
struct MsNmfProblem {
    int k;
    long long w_off;
    long long h_off;
    long long x_off;
};

__host__ __device__ inline int cd_odd(int v) { return v | 1; }  // row stride in doubles: an odd stride is free of bank conflicts

__device__ __forceinline__ double cd_warp_sum(double v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// One coordinate-descent sweep over the K entries of one row w (of W, or of H^T): G = the K x K Gram matrix (row
// stride gs), b = the K right-hand sides (XHt row, or X^T W row).  Returns the row's share of the violation.
template <int K>
__device__ __forceinline__ double cd_row_sweep(double (&w)[K], const double (&b)[K], const double* G, int gs) {
    double viol = 0.0;
#pragma unroll
    for (int t = 0; t < K; t++) {
        double grad = -b[t];
#pragma unroll
        for (int r = 0; r < K; r++) grad = fma(G[t * gs + r], w[r], grad);
        viol += fabs(w[t] == 0.0 ? fmin(0.0, grad) : grad);
        const double hess = G[t * gs + t];
        if (hess != 0.0) w[t] = fmax(w[t] - grad / hess, 0.0);
    }
    return viol;
}

// Output e of [W^T W (K x K) | W^T X (K x m)] summed over rows s, s + slices, ... < rows of a tile in shared memory
// (sW rows ws apart, sX rows xs apart).  With K = m and sW = sX this is X^T X.
__device__ __forceinline__ double cd_gram_item(int e, int s, int slices, int rows, const double* sW, int ws, int K,
                                               const double* sX, int xs, int m) {
    const double *a, *b;
    int bs;
    if (e < K * K) {
        a = sW + e / K;
        b = sW + e % K;
        bs = ws;
    } else {
        e -= K * K;
        a = sW + e / m;
        b = sX + e % m;
        bs = xs;
    }
    double acc0 = 0.0, acc1 = 0.0;  // two chains: each product waits on a shared-memory load
    int i = s;
    for (; i + slices < rows; i += 2 * slices) {
        acc0 = fma(a[i * ws], b[i * bs], acc0);
        acc1 = fma(a[(i + slices) * ws], b[(i + slices) * bs], acc1);
    }
    if (i < rows) acc0 = fma(a[i * ws], b[i * bs], acc0);
    return acc0 + acc1;
}

__host__ __device__ inline int cd_slices(int n_out, int rows) {
    int s = CD_THREADS / n_out;
    if (s < 1) s = 1;
    if (s > rows) s = rows;
    return s;
}

// ---------------------------------------------------------------------------------------------------
// resident regime
// ---------------------------------------------------------------------------------------------------
// Shared memory (doubles): sX [n][XS], sW [n][WS], sH [K][m], sHHt [K][K], sWtW [K][K], sWtX [K][m],
// sPart [max(CD_THREADS, n_out)], s_red [2][32]
template <int K>
__device__ __forceinline__ void cd_resident_body(const double* __restrict__ X, int n, int m, double* __restrict__ Wp,
                                                 double* __restrict__ Hp, int max_iter, double tol, int32_t* n_iter_out,
                                                 double* err_out, double* vaf_out, double* sm) {
    const int XS = cd_odd(m), WS = cd_odd(K);
    const int n_out = K * K + K * m, slices = cd_slices(n_out, n), n_items = n_out * slices;
    double* sX = sm;
    double* sW = sX + n * XS;
    double* sH = sW + n * WS;
    double* sHHt = sH + K * m;
    double* sWtW = sHHt + K * K;
    double* sWtX = sWtW + K * K;
    double* sPart = sWtX + K * m;
    double* s_red = sPart + (n_out > CD_THREADS ? n_out : CD_THREADS);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    for (int i = tid; i < n * m; i += CD_THREADS) sX[(i / m) * XS + i % m] = X[i];
    for (int i = tid; i < n * K; i += CD_THREADS) sW[(i / K) * WS + i % K] = Wp[i];
    for (int i = tid; i < K * m; i += CD_THREADS) sH[i] = Hp[i];
    __syncthreads();

    double viol_init = 0.0;
    int it = 0;
    for (it = 1; it <= max_iter; it++) {
        // ---- H H^T of the current H
        for (int e = tid; e < K * K; e += CD_THREADS) {
            const int a = e / K, b = e % K;
            double acc = 0.0;
            for (int j = 0; j < m; j++) acc = fma(sH[a * m + j], sH[b * m + j], acc);
            sHHt[e] = acc;
        }
        __syncthreads();
        // ---- W step: one row per thread
        double vw = 0.0;
        for (int i = tid; i < n; i += CD_THREADS) {
            double w[K], xht[K];
#pragma unroll
            for (int t = 0; t < K; t++) w[t] = sW[i * WS + t], xht[t] = 0.0;
            for (int j = 0; j < m; j++) {
                const double x = sX[i * XS + j];
#pragma unroll
                for (int t = 0; t < K; t++) xht[t] = fma(x, sH[t * m + j], xht[t]);
            }
            vw += cd_row_sweep<K>(w, xht, sHHt, K);
#pragma unroll
            for (int t = 0; t < K; t++) sW[i * WS + t] = w[t];
        }
        vw = cd_warp_sum(vw);
        if (lane == 0) s_red[warp] = vw;
        __syncthreads();
        // ---- W^T W and W^T X of the updated W: row slices side by side, then one sum per output
        for (int item = tid; item < n_items; item += CD_THREADS)
            sPart[item] = cd_gram_item(item % n_out, item / n_out, slices, n, sW, WS, K, sX, XS, m);
        __syncthreads();
        for (int e = tid; e < n_out; e += CD_THREADS) {
            double acc = 0.0;
            for (int s = 0; s < slices; s++) acc += sPart[s * n_out + e];
            if (e < K * K) sWtW[e] = acc;
            else sWtX[e - K * K] = acc;
        }
        double violation = 0.0;
        for (int w = 0; w < CD_THREADS / 32; w++) violation += s_red[w];
        __syncthreads();
        // ---- H step: one column of H per thread
        double vh = 0.0;
        if (tid < m) {
            double h[K], xtw[K];
#pragma unroll
            for (int t = 0; t < K; t++) h[t] = sH[t * m + tid], xtw[t] = sWtX[t * m + tid];
            vh = cd_row_sweep<K>(h, xtw, sWtW, K);
#pragma unroll
            for (int t = 0; t < K; t++) sH[t * m + tid] = h[t];
        }
        if (tid < 64) {  // m <= 64: the violation of the H step lives in the first two warps
            vh = cd_warp_sum(vh);
            if (lane == 0) s_red[32 + warp] = vh;
        }
        __syncthreads();
        violation += s_red[32] + s_red[33];  // sklearn: violation = 0; += W step; += H step
        if (it == 1) viol_init = violation;
        if (viol_init == 0.0 || violation / viol_init <= tol) break;
    }
    if (it > max_iter) it = max_iter;

    // ---- results: factors, ||X - W H||_F, variance accounted for (analysis.py:642-667)
    for (int i = tid; i < n * K; i += CD_THREADS) Wp[i] = sW[(i / K) * WS + i % K];
    for (int i = tid; i < K * m; i += CD_THREADS) Hp[i] = sH[i];
    // per column: residual and total sums of squares, one column per thread
    for (int j = tid; j < m; j += CD_THREADS) {
        double rs = 0.0, cs = 0.0;
        for (int i = 0; i < n; i++) {
            double r = sX[i * XS + j];
            cs = fma(r, r, cs);
#pragma unroll
            for (int c = 0; c < K; c++) r = fma(-sW[i * WS + c], sH[c * m + j], r);
            rs = fma(r, r, rs);
        }
        sPart[j] = rs;
        sPart[CD_MAX_M + j] = cs;
        vaf_out[1 + j] = 1.0 - rs / cs;
    }
    __syncthreads();
    if (tid == 0) {
        double rs = 0.0, cs = 0.0;
        for (int j = 0; j < m; j++) rs += sPart[j], cs += sPart[CD_MAX_M + j];
        *n_iter_out = it;
        *err_out = sqrt(rs);
        vaf_out[0] = 1.0 - rs / cs;
    }
}

#define CD_K_SWITCH(KEXPR, CALL)                                                                                      \
    switch (KEXPR) {                                                                                                  \
        case 1: CALL(1); break;   case 2: CALL(2); break;   case 3: CALL(3); break;   case 4: CALL(4); break;         \
        case 5: CALL(5); break;   case 6: CALL(6); break;   case 7: CALL(7); break;   case 8: CALL(8); break;         \
        case 9: CALL(9); break;   case 10: CALL(10); break; case 11: CALL(11); break; case 12: CALL(12); break;       \
        case 13: CALL(13); break; case 14: CALL(14); break; case 15: CALL(15); break; case 16: CALL(16); break;       \
        default: break;                                                                                               \
    }

__global__ void __launch_bounds__(CD_THREADS)
    ms_cd_resident_kernel(const double* __restrict__ X, int n, int m, const MsNmfProblem* __restrict__ problems,
                          double* __restrict__ Wg, double* __restrict__ Hg, int max_iter, double tol,
                          int32_t* __restrict__ n_iter_out, double* __restrict__ err_out, double* __restrict__ vaf_out) {
    extern __shared__ double cd_sm[];
    const MsNmfProblem pb = problems[blockIdx.x];
    const int p = blockIdx.x;
#define CD_RESIDENT(KK)                                                                                               \
    cd_resident_body<KK>(X + pb.x_off, n, m, Wg + pb.w_off, Hg + pb.h_off, max_iter, tol, n_iter_out + p, err_out + p, \
                         vaf_out + (long long)p * (m + 1), cd_sm)
    CD_K_SWITCH(pb.k, CD_RESIDENT)
#undef CD_RESIDENT
}

static size_t cd_resident_fixed(int m, int kmax) {
    const int n_out = kmax * kmax + kmax * m;
    return (size_t)kmax * m * 2 + (size_t)kmax * kmax * 2 + (size_t)(n_out > CD_THREADS ? n_out : CD_THREADS) + 64;
}
static size_t cd_resident_row(int m, int kmax) { return (size_t)cd_odd(m) + (size_t)cd_odd(kmax); }

// Largest n the resident CD kernel takes for (m, kmax); 0 if the shape is unsupported.
extern "C" int32_t ms_nmf_cd_resident_max_rows(int32_t m, int32_t kmax) {
    if (m < 1 || m > CD_MAX_M || kmax < 1 || kmax > CD_MAX_K) return 0;
    const size_t budget = 227 * 1024 - 1024;
    const size_t fixed = sizeof(double) * cd_resident_fixed(m, kmax);
    // the row slices of the Gram reduction (<= n_out * slices partials) must fit the partial buffer: n_out * slices <=
    // max(CD_THREADS, n_out) holds for every n by construction of cd_slices
    return (int32_t)((budget - fixed) / (sizeof(double) * cd_resident_row(m, kmax)));
}

extern "C" int ms_nmf_cd_batched_planned(const double* d_X, int32_t n, int32_t m, const void* d_table, int32_t n_problems,
                                         int32_t kmax, double* d_W, double* d_H, int32_t max_iter, double tol,
                                         int32_t* d_n_iter, double* d_err, double* d_vaf, void* stream) {
    if (!d_X || !d_table || !d_W || !d_H || !d_n_iter || !d_err || !d_vaf) return MS_E_INVALID;
    if (n < 1 || m < 1 || m > CD_MAX_M || kmax < 1 || kmax > CD_MAX_K || n_problems < 0 || max_iter < 0 || !(tol >= 0.0))
        return MS_E_INVALID;
    if (n_problems == 0) return MS_OK;
    if (n > ms_nmf_cd_resident_max_rows(m, kmax)) return MS_E_INVALID;  // too long for shared memory: ms_nmf_cd_stream
    const size_t smem = sizeof(double) * ((size_t)n * cd_resident_row(m, kmax) + cd_resident_fixed(m, kmax));
    MS_CUDA_CHECK(cudaFuncSetAttribute(ms_cd_resident_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ms_cd_resident_kernel<<<n_problems, CD_THREADS, smem, (cudaStream_t)stream>>>(
        d_X, n, m, (const MsNmfProblem*)d_table, d_W, d_H, max_iter, tol, d_n_iter, d_err, d_vaf);
    MS_COUNT_LAUNCH();
    MS_CUDA_CHECK(cudaGetLastError());
    return MS_OK;
}

// ---------------------------------------------------------------------------------------------------
// streaming regime
// ---------------------------------------------------------------------------------------------------
#define CDS_ROWS CD_THREADS

struct MsCdStreamState {  // per problem, device memory
    double HHt[CD_MAX_K * CD_MAX_K];
    double acc[CD_MAX_K * CD_MAX_K + CD_MAX_K * CD_MAX_M];  // W^T W [K][K], then W^T X [K][m]
    double viol_w;                                          // violation of the W step (atomics of the W pass)
    double viol_init;
    int n_iter, done;
};

// One pass over X and W of one problem: per 256-row tile, X and W rows are staged in shared memory (coalesced),
// each thread runs the W step of one row, the tile goes back, and its share of W^T W / W^T X is added to register
// accumulators that live across every tile the CTA visits; one atomicAdd per CTA and output at the end.
template <int K>
__device__ __forceinline__ void cd_stream_w_body(const double* __restrict__ X, long long n, int m, double* __restrict__ Wp,
                                                 const double* __restrict__ Hp, MsCdStreamState* __restrict__ st,
                                                 double* sm) {
    const int XS = cd_odd(m), WS = cd_odd(K);
    const int n_out = K * K + K * m, slices = cd_slices(n_out, CDS_ROWS), n_items = n_out * slices;
    double* sX = sm;                     // [CDS_ROWS][XS]
    double* sW = sX + CDS_ROWS * XS;     // [CDS_ROWS][WS]
    double* sH = sW + CDS_ROWS * WS;     // [K][m]
    double* sHHt = sH + K * m;           // [K][K]
    double* s_red = sHHt + K * K;        // [32]
    const int tid = threadIdx.x;
    for (int i = tid; i < K * m; i += CDS_ROWS) sH[i] = Hp[i];
    for (int i = tid; i < K * K; i += CDS_ROWS) sHHt[i] = st->HHt[i];
    double acc[CD_ITEMS];
#pragma unroll
    for (int q = 0; q < CD_ITEMS; q++) acc[q] = 0.0;
    double vw = 0.0;
    const long long n_tiles = (n + CDS_ROWS - 1) / CDS_ROWS;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const long long r0 = tile * CDS_ROWS;
        const int rows = (int)min((long long)CDS_ROWS, n - r0);
        __syncthreads();  // the previous tile's reductions are done with the buffers
        for (int i = tid; i < rows * m; i += CDS_ROWS) sX[(i / m) * XS + i % m] = X[r0 * m + i];
        for (int i = tid; i < rows * K; i += CDS_ROWS) sW[(i / K) * WS + i % K] = Wp[r0 * K + i];
        __syncthreads();
        if (tid < rows) {
            double w[K], xht[K];
#pragma unroll
            for (int t = 0; t < K; t++) w[t] = sW[tid * WS + t], xht[t] = 0.0;
            for (int j = 0; j < m; j++) {
                const double x = sX[tid * XS + j];
#pragma unroll
                for (int t = 0; t < K; t++) xht[t] = fma(x, sH[t * m + j], xht[t]);
            }
            vw += cd_row_sweep<K>(w, xht, sHHt, K);
#pragma unroll
            for (int t = 0; t < K; t++) sW[tid * WS + t] = w[t];
        }
        __syncthreads();
        for (int i = tid; i < rows * K; i += CDS_ROWS) Wp[r0 * K + i] = sW[(i / K) * WS + i % K];
        const int sl = cd_slices(n_out, rows);  // == slices except in a short last tile
#pragma unroll
        for (int q = 0; q < CD_ITEMS; q++) {
            const int item = tid + q * CDS_ROWS;
            if (item < n_items) {
                const int s = item / n_out;
                if (s < sl) acc[q] += cd_gram_item(item % n_out, s, sl, rows, sW, WS, K, sX, XS, m);
            }
        }
    }
#pragma unroll
    for (int q = 0; q < CD_ITEMS; q++) {
        const int item = tid + q * CDS_ROWS;
        if (item < n_items) atomicAdd(&st->acc[item % n_out], acc[q]);
    }
    vw = cd_warp_sum(vw);
    if ((tid & 31) == 0) s_red[tid >> 5] = vw;
    __syncthreads();
    if (tid == 0) {
        double v = 0.0;
        for (int w = 0; w < CDS_ROWS / 32; w++) v += s_red[w];
        atomicAdd(&st->viol_w, v);
    }
}

__global__ void __launch_bounds__(CDS_ROWS)
    ms_cd_stream_w_kernel(const double* __restrict__ X, long long n, int m, const MsNmfProblem* __restrict__ problems,
                          double* __restrict__ Wg, const double* __restrict__ Hg, MsCdStreamState* __restrict__ states) {
    extern __shared__ double cd_sm[];
    const MsNmfProblem pb = problems[blockIdx.y];
    MsCdStreamState* st = states + blockIdx.y;
    if (st->done) return;
#define CD_STREAM_W(KK) cd_stream_w_body<KK>(X + pb.x_off, n, m, Wg + pb.w_off, Hg + pb.h_off, st, cd_sm)
    CD_K_SWITCH(pb.k, CD_STREAM_W)
#undef CD_STREAM_W
}

// mode 0: prepare (H H^T of the initial H, clear the accumulators); mode 1: H step and stop test after a W pass
__global__ void __launch_bounds__(64)
    ms_cd_stream_h_kernel(int m, const MsNmfProblem* __restrict__ problems, double* __restrict__ Hg,
                          MsCdStreamState* __restrict__ states, int mode, int iteration, double tol) {
    __shared__ double sH[CD_MAX_K * CD_MAX_M];
    __shared__ double s_red[2];
    const MsNmfProblem pb = problems[blockIdx.x];
    MsCdStreamState* st = states + blockIdx.x;
    const int k = pb.k, tid = threadIdx.x;
    double* Hp = Hg + pb.h_off;
    if (mode == 1 && st->done) return;
    for (int e = tid; e < k * m; e += 64) sH[e] = Hp[e];
    __syncthreads();
    if (mode == 0) {
        if (tid == 0) st->done = 0, st->n_iter = 0, st->viol_init = 0.0;
    } else {
        // the column sweep of cd_row_sweep with a run-time k (one small CTA per problem; not on the critical path)
        const double* WtW = st->acc;
        const double* WtX = st->acc + k * k;
        double vh = 0.0;
        if (tid < m) {
            for (int t = 0; t < k; t++) {
                double grad = -WtX[t * m + tid];
                for (int r = 0; r < k; r++) grad = fma(WtW[t * k + r], sH[r * m + tid], grad);
                const double h = sH[t * m + tid];
                vh += fabs(h == 0.0 ? fmin(0.0, grad) : grad);
                const double hess = WtW[t * k + t];
                if (hess != 0.0) sH[t * m + tid] = fmax(h - grad / hess, 0.0);
            }
        }
        vh = cd_warp_sum(vh);
        if ((tid & 31) == 0) s_red[tid >> 5] = vh;
        __syncthreads();
        for (int e = tid; e < k * m; e += 64) Hp[e] = sH[e];
        if (tid == 0) {
            const double violation = st->viol_w + (s_red[0] + s_red[1]);
            if (iteration == 1) st->viol_init = violation;
            st->n_iter = iteration;
            if (st->viol_init == 0.0 || violation / st->viol_init <= tol) st->done = 1;
        }
    }
    for (int e = tid; e < k * k; e += 64) {
        const int a = e / k, b = e % k;
        double acc = 0.0;
        for (int j = 0; j < m; j++) acc = fma(sH[a * m + j], sH[b * m + j], acc);
        st->HHt[e] = acc;
    }
    __syncthreads();  // every thread has read the accumulators (H step) before they are cleared
    for (int e = tid; e < k * k + k * m; e += 64) st->acc[e] = 0.0;
    if (tid == 0) st->viol_w = 0.0;
}

// per problem and column: sum of squares of the residual X - W H and of X (sums: [P][2][m]), for err and VAF
__global__ void __launch_bounds__(256)
    ms_cd_stream_vaf_kernel(const double* __restrict__ X, long long n, int m, const MsNmfProblem* __restrict__ problems,
                            const double* __restrict__ Wg, const double* __restrict__ Hg, double* __restrict__ sums) {
    __shared__ double sH[CD_MAX_K * CD_MAX_M];
    const MsNmfProblem pb = problems[blockIdx.y];
    const int k = pb.k;
    const double* Xp = X + pb.x_off;
    const double* Wp = Wg + pb.w_off;
    for (int e = threadIdx.x; e < k * m; e += 256) sH[e] = Hg[pb.h_off + e];
    __syncthreads();
    const int j = threadIdx.x % m, lane_row = threadIdx.x / m, rows_per_pass = 256 / m;
    if (lane_row >= rows_per_pass) return;
    double rs = 0.0, cs = 0.0;
    for (long long i = (long long)blockIdx.x * rows_per_pass + lane_row; i < n; i += (long long)gridDim.x * rows_per_pass) {
        double r = Xp[i * m + j];
        cs = fma(r, r, cs);
        for (int c = 0; c < k; c++) r = fma(-Wp[i * k + c], sH[c * m + j], r);
        rs = fma(r, r, rs);
    }
    atomicAdd(&sums[((long long)blockIdx.y * 2 + 0) * m + j], rs);
    atomicAdd(&sums[((long long)blockIdx.y * 2 + 1) * m + j], cs);
}

__global__ void ms_cd_stream_finish_kernel(int m, const MsCdStreamState* __restrict__ states, const double* __restrict__ sums,
                                           int32_t* __restrict__ n_iter, double* __restrict__ err, double* __restrict__ vaf) {
    const int p = blockIdx.x;
    const double* rs_col = sums + (long long)p * 2 * m;
    const double* cs_col = rs_col + m;
    for (int j = threadIdx.x; j < m; j += blockDim.x) vaf[(long long)p * (m + 1) + 1 + j] = 1.0 - rs_col[j] / cs_col[j];
    if (threadIdx.x == 0) {
        double rs = 0.0, cs = 0.0;
        for (int j = 0; j < m; j++) rs += rs_col[j], cs += cs_col[j];
        vaf[(long long)p * (m + 1)] = 1.0 - rs / cs;
        err[p] = sqrt(rs);
        n_iter[p] = states[p].n_iter;
    }
}

static size_t cd_align256(size_t b) { return (b + 255) / 256 * 256; }

extern "C" int64_t ms_nmf_cd_stream_workspace_bytes(int32_t m, int32_t n_problems) {
    if (m < 1 || n_problems < 0) return 0;
    return (int64_t)(cd_align256(sizeof(MsCdStreamState) * (size_t)n_problems) + sizeof(double) * 2 * (size_t)m * n_problems +
                     256);
}

extern "C" int ms_nmf_cd_stream(const double* d_X, int64_t n, int32_t m, const void* d_table, int32_t n_problems,
                                int32_t kmax, double* d_W, double* d_H, int32_t max_iter, double tol, void* d_work,
                                int32_t* d_n_iter, double* d_err, double* d_vaf, void* stream) {
    if (!d_X || !d_table || !d_W || !d_H || !d_work || !d_n_iter || !d_err || !d_vaf) return MS_E_INVALID;
    if (n < 1 || m < 1 || m > CD_MAX_M || kmax < 1 || kmax > CD_MAX_K || n_problems < 0 || max_iter < 0 || !(tol >= 0.0))
        return MS_E_INVALID;
    if (n_problems == 0) return MS_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const MsNmfProblem* d_problems = (const MsNmfProblem*)d_table;
    MsCdStreamState* d_states = (MsCdStreamState*)d_work;
    double* d_sums = (double*)((char*)d_work + cd_align256(sizeof(MsCdStreamState) * (size_t)n_problems));
    MS_CUDA_CHECK(cudaMemsetAsync(d_states, 0, sizeof(MsCdStreamState) * (size_t)n_problems, st));

    const long long n_tiles = (n + CDS_ROWS - 1) / CDS_ROWS;
    long long ctas = (148LL * 4 + n_problems - 1) / n_problems;  // about one wave of the W pass over all problems
    if (ctas > n_tiles) ctas = n_tiles;
    const size_t smem = sizeof(double) * ((size_t)CDS_ROWS * (cd_odd(m) + cd_odd(kmax)) + (size_t)kmax * m + kmax * kmax + 32);
    MS_CUDA_CHECK(cudaFuncSetAttribute(ms_cd_stream_w_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ms_cd_stream_h_kernel<<<n_problems, 64, 0, st>>>(m, d_problems, d_H, d_states, 0, 0, tol);
    MS_COUNT_LAUNCH();
    int32_t* h_done = (int32_t*)malloc(sizeof(MsCdStreamState) * (size_t)n_problems);
    if (!h_done) return MS_E_INVALID;
    for (int it = 1; it <= max_iter; it++) {
        ms_cd_stream_w_kernel<<<dim3((unsigned)ctas, n_problems), CDS_ROWS, smem, st>>>(d_X, n, m, d_problems, d_W, d_H, d_states);
        MS_COUNT_LAUNCH();
        ms_cd_stream_h_kernel<<<n_problems, 64, 0, st>>>(m, d_problems, d_H, d_states, 1, it, tol);
        MS_COUNT_LAUNCH();
        if (it % 64 == 0 && it < max_iter) {
            // stop early once every problem has converged (pageable copy: waits for the stream)
            cudaError_t e = cudaMemcpyAsync(h_done, d_states, sizeof(MsCdStreamState) * (size_t)n_problems,
                                            cudaMemcpyDeviceToHost, st);
            if (e == cudaSuccess) e = cudaStreamSynchronize(st);
            if (e != cudaSuccess) {
                free(h_done);
                MS_CUDA_CHECK(e);
            }
            const MsCdStreamState* hs = (const MsCdStreamState*)h_done;
            int all_done = 1;
            for (int p = 0; p < n_problems; p++) all_done &= hs[p].done != 0;
            if (all_done) break;
        }
    }
    free(h_done);
    const int vaf_rows = 256 / m;
    long long vaf_ctas = (148LL * 8 + n_problems - 1) / n_problems, vaf_cap = (n + vaf_rows - 1) / vaf_rows;
    if (vaf_ctas > vaf_cap) vaf_ctas = vaf_cap;
    MS_CUDA_CHECK(cudaMemsetAsync(d_sums, 0, sizeof(double) * 2 * (size_t)m * n_problems, st));
    ms_cd_stream_vaf_kernel<<<dim3((unsigned)vaf_ctas, n_problems), 256, 0, st>>>(d_X, n, m, d_problems, d_W, d_H, d_sums);
    MS_COUNT_LAUNCH();
    ms_cd_stream_finish_kernel<<<n_problems, 64, 0, st>>>(m, d_states, d_sums, d_n_iter, d_err, d_vaf);
    MS_COUNT_LAUNCH();
    MS_CUDA_CHECK(cudaGetLastError());
    return MS_OK;
}

// ---------------------------------------------------------------------------------------------------
// NNDSVD initialisation (_initialize_nmf, init="nndsvd" / "nndsvda") from an exact SVD
// ---------------------------------------------------------------------------------------------------
// Workspace per distinct matrix b of the stack (doubles): G [m][m] (X^T X), V [m][m] (right singular vectors,
// column j = j-th largest), S [m] (singular values; 0 where the matrix is numerically rank deficient),
// U2 [2][CD_MAX_K] (squared norms of the positive / negative parts of U[:, j] = X V[:, j] / S[j]), sum (of X).
struct MsNndsvdMatrix {
    double G[CD_MAX_M * CD_MAX_M];
    double V[CD_MAX_M * CD_MAX_M];
    double S[CD_MAX_M];
    double U2[2][CD_MAX_K];
    double sum;
};

// pass 1 over X: X^T X and the sum of X, per matrix (grid.y)
__global__ void __launch_bounds__(CDS_ROWS)
    ms_nndsvd_gram_kernel(const double* __restrict__ X, long long n, int m, MsNndsvdMatrix* __restrict__ mats) {
    extern __shared__ double cd_sm[];
    const int XS = cd_odd(m), n_out = m * m, tid = threadIdx.x;
    const double* Xb = X + (long long)blockIdx.y * n * m;
    MsNndsvdMatrix* mt = mats + blockIdx.y;
    double* sX = cd_sm;                  // [CDS_ROWS][XS]
    double* s_red = sX + CDS_ROWS * XS;  // [32]
    double acc[CD_MAX_M * CD_MAX_M / CD_THREADS];
#pragma unroll
    for (int q = 0; q < CD_MAX_M * CD_MAX_M / CD_THREADS; q++) acc[q] = 0.0;
    const int slices = cd_slices(n_out, CDS_ROWS), n_items = n_out * slices;
    double total = 0.0;
    const long long n_tiles = (n + CDS_ROWS - 1) / CDS_ROWS;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const long long r0 = tile * CDS_ROWS;
        const int rows = (int)min((long long)CDS_ROWS, n - r0);
        __syncthreads();
        for (int i = tid; i < rows * m; i += CDS_ROWS) {
            const double v = Xb[r0 * m + i];
            sX[(i / m) * XS + i % m] = v;
            total += v;
        }
        __syncthreads();
        const int sl = cd_slices(n_out, rows);
#pragma unroll
        for (int q = 0; q < CD_MAX_M * CD_MAX_M / CD_THREADS; q++) {
            const int item = tid + q * CDS_ROWS;
            if (item < n_items && item / n_out < sl) acc[q] += cd_gram_item(item % n_out, item / n_out, sl, rows, sX, XS, m, sX, XS, m);
        }
    }
#pragma unroll
    for (int q = 0; q < CD_MAX_M * CD_MAX_M / CD_THREADS; q++) {
        const int item = tid + q * CDS_ROWS;
        if (item < n_items) atomicAdd(&mt->G[item % n_out], acc[q]);
    }
    total = cd_warp_sum(total);
    if ((tid & 31) == 0) s_red[tid >> 5] = total;
    __syncthreads();
    if (tid == 0) {
        double v = 0.0;
        for (int w = 0; w < CDS_ROWS / 32; w++) v += s_red[w];
        atomicAdd(&mt->sum, v);
    }
}

// Eigen-decomposition of G = X^T X by cyclic Jacobi rotations, one warp per matrix; S = sqrt of the eigenvalues in
// descending order, V their eigenvectors.  An eigenvalue at or below m * eps * the largest one is treated as zero.
__global__ void __launch_bounds__(32) ms_nndsvd_eig_kernel(int m, MsNndsvdMatrix* __restrict__ mats) {
    __shared__ double A[CD_MAX_M * (CD_MAX_M + 1)];
    __shared__ int order[CD_MAX_M];
    MsNndsvdMatrix* mt = mats + blockIdx.x;
    const int lane = threadIdx.x, AS = CD_MAX_M + 1, VS = m;
    double* V = mt->G;  // G is read into A first; its storage then accumulates the rotations
    for (int e = lane; e < m * m; e += 32) {
        const int r = e / m, c = e % m;
        A[r * AS + c] = 0.5 * (mt->G[r * m + c] + mt->G[c * m + r]);  // symmetric up to the atomics' summation order
    }
    __syncwarp();
    for (int e = lane; e < m * m; e += 32) V[e] = (e / m == e % m) ? 1.0 : 0.0;
    __syncwarp();
    // a sweep rotates every pair whose off-diagonal entry is not negligible next to its diagonal entries (the test of
    // Demmel and Veselic, which keeps small eigenvalues to high relative accuracy); a sweep without rotation ends it
    for (int sweep = 0; sweep < 60; sweep++) {
        int rotations = 0;
        for (int p = 0; p < m - 1; p++) {
            for (int q = p + 1; q < m; q++) {
                const double apq = A[p * AS + q];
                // uniform across the warp: every lane read the same values
                if (!(fabs(apq) > 2.220446049250313e-16 * sqrt(fabs(A[p * AS + p] * A[q * AS + q])))) continue;
                rotations++;
                const double theta = (A[q * AS + q] - A[p * AS + p]) / (2.0 * apq);
                const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
                const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
                __syncwarp();
                for (int r = lane; r < m; r += 32) {  // A <- A J
                    const double arp = A[r * AS + p], arq = A[r * AS + q];
                    A[r * AS + p] = c * arp - s * arq;
                    A[r * AS + q] = s * arp + c * arq;
                    const double vrp = V[r * VS + p], vrq = V[r * VS + q];
                    V[r * VS + p] = c * vrp - s * vrq;
                    V[r * VS + q] = s * vrp + c * vrq;
                }
                __syncwarp();
                for (int r = lane; r < m; r += 32) {  // A <- J^T A
                    const double apr = A[p * AS + r], aqr = A[q * AS + r];
                    A[p * AS + r] = c * apr - s * aqr;
                    A[q * AS + r] = s * apr + c * aqr;
                }
                __syncwarp();
            }
        }
        if (rotations == 0) break;
    }
    if (lane == 0) {
        for (int j = 0; j < m; j++) order[j] = j;
        for (int j = 0; j < m; j++) {  // selection sort, descending eigenvalue (stable: ties keep index order)
            int best = j;
            for (int r = j + 1; r < m; r++)
                if (A[order[r] * AS + order[r]] > A[order[best] * AS + order[best]]) best = r;
            const int tmp = order[j];
            order[j] = order[best];
            order[best] = tmp;
        }
    }
    __syncwarp();
    const double lmax = A[order[0] * AS + order[0]];
    for (int j = lane; j < m; j += 32) {
        const double l = A[order[j] * AS + order[j]];
        mt->S[j] = (l > (double)m * 2.220446049250313e-16 * lmax && l > 0.0) ? sqrt(l) : 0.0;
    }
    for (int e = lane; e < m * m; e += 32) {
        const int r = e / m, j = e % m;
        mt->V[r * m + j] = V[r * VS + order[j]];
    }
    for (int e = lane; e < 2 * CD_MAX_K; e += 32) mt->U2[e / CD_MAX_K][e % CD_MAX_K] = 0.0;
}

// u_ij = X[i, :] . V[:, j] / S[j] for j < kk (S[j] == 0: 0, flagged by the fill kernel)
__device__ __forceinline__ void nndsvd_u_row(const double* __restrict__ xrow, int m, const double* sV, const double* sInvS,
                                             int kk, double (&u)[CD_MAX_K]) {
#pragma unroll
    for (int j = 0; j < CD_MAX_K; j++) u[j] = 0.0;
    for (int c = 0; c < m; c++) {
        const double x = xrow[c];
#pragma unroll
        for (int j = 0; j < CD_MAX_K; j++)
            if (j < kk) u[j] = fma(x, sV[c * CD_MAX_K + j], u[j]);
    }
#pragma unroll
    for (int j = 0; j < CD_MAX_K; j++) u[j] *= sInvS[j];
}

// pass 2 over X: squared norms of the positive and negative parts of the first kk left singular vectors
__global__ void __launch_bounds__(256)
    ms_nndsvd_norms_kernel(const double* __restrict__ X, long long n, int m, int kk, MsNndsvdMatrix* __restrict__ mats) {
    __shared__ double sV[CD_MAX_M * CD_MAX_K];
    __shared__ double sInvS[CD_MAX_K];
    MsNndsvdMatrix* mt = mats + blockIdx.y;
    const double* Xb = X + (long long)blockIdx.y * n * m;
    for (int e = threadIdx.x; e < m * CD_MAX_K; e += 256) sV[e] = (e % CD_MAX_K) < kk ? mt->V[(e / CD_MAX_K) * m + e % CD_MAX_K] : 0.0;
    for (int j = threadIdx.x; j < CD_MAX_K; j += 256) sInvS[j] = (j < kk && mt->S[j] > 0.0) ? 1.0 / mt->S[j] : 0.0;
    __syncthreads();
    double pos[CD_MAX_K], neg[CD_MAX_K];
#pragma unroll
    for (int j = 0; j < CD_MAX_K; j++) pos[j] = neg[j] = 0.0;
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
        double u[CD_MAX_K];
        nndsvd_u_row(Xb + i * m, m, sV, sInvS, kk, u);
#pragma unroll
        for (int j = 0; j < CD_MAX_K; j++) {
            if (u[j] > 0.0) pos[j] = fma(u[j], u[j], pos[j]);
            else neg[j] = fma(u[j], u[j], neg[j]);
        }
    }
#pragma unroll
    for (int j = 0; j < CD_MAX_K; j++) {
        if (j >= kk) break;
        const double p = cd_warp_sum(pos[j]), q = cd_warp_sum(neg[j]);
        if ((threadIdx.x & 31) == 0) {
            atomicAdd(&mt->U2[0][j], p);
            atomicAdd(&mt->U2[1][j], q);
        }
    }
}

// pass 3 over X: W and H of every problem (grid.y), sklearn's choice of the positive or the negative part for j >= 1
// (ties go to the negative part), entries below 1e-6 zeroed, and for nndsvda the zeros filled with X.mean()
__global__ void __launch_bounds__(256)
    ms_nndsvd_fill_kernel(const double* __restrict__ X, long long n, int m, const MsNmfProblem* __restrict__ problems,
                          const MsNndsvdMatrix* __restrict__ mats, int variant, double* __restrict__ Wg,
                          double* __restrict__ Hg, int32_t* __restrict__ status) {
    __shared__ double sV[CD_MAX_M * CD_MAX_K];
    __shared__ double sInvS[CD_MAX_K];
    __shared__ double sScaleU[CD_MAX_K];  // W[:, j] = sScaleU[j] * (part of u_j); sign: +1 positive part, -1 negative
    __shared__ double sSign[CD_MAX_K];
    const MsNmfProblem pb = problems[blockIdx.y];
    const int k = pb.k;
    const long long b = pb.x_off / (n * m);
    const MsNndsvdMatrix* mt = mats + b;
    const double* Xb = X + pb.x_off;
    const double avg = mt->sum / ((double)n * m);
    const double eps = 1e-6;
    for (int e = threadIdx.x; e < m * CD_MAX_K; e += 256) sV[e] = (e % CD_MAX_K) < k ? mt->V[(e / CD_MAX_K) * m + e % CD_MAX_K] : 0.0;
    for (int j = threadIdx.x; j < CD_MAX_K; j += 256) sInvS[j] = (j < k && mt->S[j] > 0.0) ? 1.0 / mt->S[j] : 0.0;
    __syncthreads();
    if (threadIdx.x < k) {
        const int j = threadIdx.x;
        double scale = 0.0, sign = 1.0;
        bool bad = !(mt->S[j] > 0.0);
        double yp2 = 0.0, yn2 = 0.0;
        for (int c = 0; c < m; c++) {
            const double v = sV[c * CD_MAX_K + j];
            if (v > 0.0) yp2 += v * v;
            else yn2 += v * v;
        }
        if (j == 0) {
            scale = sqrt(mt->S[0]);
            sign = 0.0;  // |u|, |v|
        } else {
            const double xp = sqrt(mt->U2[0][j]), xn = sqrt(mt->U2[1][j]), yp = sqrt(yp2), yn = sqrt(yn2);
            const double mp = xp * yp, mn = xn * yn;
            double xn_, yn_, sigma;
            if (mp > mn) xn_ = xp, yn_ = yp, sigma = mp, sign = 1.0;
            else xn_ = xn, yn_ = yn, sigma = mn, sign = -1.0;
            if (xn_ == 0.0 || yn_ == 0.0) bad = true;
            const double lbd = sqrt(mt->S[j] * sigma);
            scale = lbd / xn_;
            // H row j: lbd * (part of v) / its norm
            if (blockIdx.x == 0)
                for (int c = 0; c < m; c++) {
                    const double v = sign * sV[c * CD_MAX_K + j];
                    double h = v > 0.0 ? lbd * v / yn_ : 0.0;
                    if (h < eps) h = variant ? avg : 0.0;
                    Hg[pb.h_off + (long long)j * m + c] = h;
                }
        }
        if (j == 0 && blockIdx.x == 0)
            for (int c = 0; c < m; c++) {
                double h = scale * fabs(sV[c * CD_MAX_K]);
                if (h < eps) h = variant ? avg : 0.0;
                Hg[pb.h_off + c] = h;
            }
        if (bad && blockIdx.x == 0) atomicOr(status, 1);
        sScaleU[j] = scale;
        sSign[j] = sign;
    }
    __syncthreads();
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
        double u[CD_MAX_K];
        nndsvd_u_row(Xb + i * m, m, sV, sInvS, k, u);
#pragma unroll
        for (int j = 0; j < CD_MAX_K; j++) {
            if (j >= k) break;
            const double s = sSign[j];
            const double part = s == 0.0 ? fabs(u[j]) : (s * u[j] > 0.0 ? s * u[j] : 0.0);
            double w = sScaleU[j] * part;
            if (w < eps) w = variant ? avg : 0.0;
            Wg[pb.w_off + i * k + j] = w;
        }
    }
}

extern "C" int64_t ms_nndsvd_workspace_bytes(int32_t m, int32_t n_matrices) {
    if (m < 1 || n_matrices < 0) return 0;
    return (int64_t)sizeof(MsNndsvdMatrix) * n_matrices + 256;
}

extern "C" int ms_nndsvd_init(const double* d_X, int64_t n, int32_t m, int32_t n_matrices, const void* d_table,
                              int32_t n_problems, int32_t kmax, int32_t variant, void* d_work, double* d_W, double* d_H,
                              int32_t* d_status, void* stream) {
    if (!d_X || !d_table || !d_work || !d_W || !d_H || !d_status) return MS_E_INVALID;
    if (n < 1 || m < 1 || m > CD_MAX_M || n_matrices < 1 || n_problems < 0 || kmax < 1 || kmax > CD_MAX_K ||
        kmax > m || kmax > n || (variant != 0 && variant != 1))
        return MS_E_INVALID;
    if (n_problems == 0) return MS_OK;
    cudaStream_t st = (cudaStream_t)stream;
    MsNndsvdMatrix* mats = (MsNndsvdMatrix*)d_work;
    MS_CUDA_CHECK(cudaMemsetAsync(mats, 0, sizeof(MsNndsvdMatrix) * (size_t)n_matrices, st));
    MS_CUDA_CHECK(cudaMemsetAsync(d_status, 0, sizeof(int32_t), st));
    const long long n_tiles = (n + CDS_ROWS - 1) / CDS_ROWS;
    long long ctas = (148LL * 4 + n_matrices - 1) / n_matrices;
    if (ctas > n_tiles) ctas = n_tiles;
    const size_t smem = sizeof(double) * ((size_t)CDS_ROWS * cd_odd(m) + 32);
    MS_CUDA_CHECK(cudaFuncSetAttribute(ms_nndsvd_gram_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ms_nndsvd_gram_kernel<<<dim3((unsigned)ctas, n_matrices), CDS_ROWS, smem, st>>>(d_X, n, m, mats);
    MS_COUNT_LAUNCH();
    ms_nndsvd_eig_kernel<<<n_matrices, 32, 0, st>>>(m, mats);
    MS_COUNT_LAUNCH();
    long long row_ctas = (n + 255) / 256, cap = (148LL * 8 + n_matrices - 1) / n_matrices;
    ms_nndsvd_norms_kernel<<<dim3((unsigned)(row_ctas < cap ? row_ctas : cap), n_matrices), 256, 0, st>>>(d_X, n, m, kmax, mats);
    MS_COUNT_LAUNCH();
    cap = (148LL * 8 + n_problems - 1) / n_problems;
    ms_nndsvd_fill_kernel<<<dim3((unsigned)(row_ctas < cap ? row_ctas : cap), n_problems), 256, 0, st>>>(
        d_X, n, m, (const MsNmfProblem*)d_table, mats, variant, d_W, d_H, d_status);
    MS_COUNT_LAUNCH();
    MS_CUDA_CHECK(cudaGetLastError());
    return MS_OK;
}
