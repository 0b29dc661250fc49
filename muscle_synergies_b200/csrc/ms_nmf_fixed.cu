// NMF with fixed synergies (H): fit W >= 0 to X for a batch of problems, fp64 - what NMF.transform does.
//
// scikit-learn 1.9.0's transform is _fit_transform(X, H=components_, update_H=False) (sklearn/decomposition/_nmf.py):
//
//   cd   W0 = 0; one _update_cdnmf_fast sweep over W per iteration (t outer, i inner):
//          grad = -XHt[i,t] + sum_r HHt[t,r] W[i,r];  violation += |grad| (|min(0, grad)| where W[i,t] == 0)
//          W[i,t] = max(W[i,t] - grad / HHt[t,t], 0) when HHt[t,t] != 0
//        stop when violation_init (iteration 1) == 0 or violation / violation_init <= tol
//   mu   W0 = sqrt(X.mean() / k) (the caller fills it); per iteration W *= XHt / (W HHt), a zero denominator replaced
//        by float32 eps; with tol > 0, every 10 iterations err = ||X - W H||_F, stop when
//        (previous err - err) / err_at_init < tol (an all-zero X makes that NaN: the loop then runs to max_iter)
//
// With H fixed, HHt and XHt are constants and the rows of W are independent: only the stop test couples them.  So
// one thread owns a row, and the same row functions (fx_xht_row, fx_cd_row, fx_mu_row, fx_mu_row_err) and the same
// H H^T (fx_hht) serve both regimes - at tol = 0 they give bit-identical W.
//
//   ms_fx_resident_kernel   one CTA per problem: X, W, XHt, HHt (and the rows' ||x_i||^2) in shared memory;
//                           iterations outer, rows inner, one fixed-order CTA reduction per stop test
//   ms_fx_chunk_kernel      long signals: rows outer, FX_CHUNK iterations inner with the row in registers; X is read
//   ms_fx_decide_kernel     once per launch (first chunk) to form XHt and ||x_i||^2, kept in the workspace;
//   ms_fx_replay_kernel     per-CTA per-iteration partial sums go to the workspace, the decide kernel reduces them in
//                           a fixed order and finds the first iteration of the chunk where the stop test fires, and
//                           the rows of a problem that stopped replay from the chunk's saved W up to it
//   ms_fx_vaf_kernel        ||X - W H|| per column, CTA partials, then ms_fx_finish_kernel sums them in a fixed order
//
// Every reduction behind a stop decision or an output has a fixed order (no floating-point atomics): two identical
// calls give bit-identical W, n_iter, err and VAF.
#include "ms_nmf_common.cuh"

#define FX_THREADS 256
#define FX_CHUNK 32                                  // iterations a streaming row runs in registers per launch
#define FX_MU_EPS 1.1920928955078125e-07             // np.finfo(np.float32).eps, sklearn's EPSILON
#define FX_SOLVER_CD 0
#define FX_SOLVER_MU 1

// ---------------------------------------------------------------------------------------------------
// per-row functions shared by both regimes
// ---------------------------------------------------------------------------------------------------
// H H^T into G[K][K] (row stride K), one output per thread, products in column order
template <int K>
__device__ __forceinline__ void fx_hht(const double* sH, int m, double* G) {
    for (int e = threadIdx.x; e < K * K; e += blockDim.x) {
        const int a = e / K, b = e % K;
        double acc = 0.0;
        for (int j = 0; j < m; j++) acc = fma(sH[a * m + j], sH[b * m + j], acc);
        G[e] = acc;
    }
}

// row i of X H^T and ||x_i||^2; X element (i, j) at x[j * cs]
template <int K>
__device__ __forceinline__ void fx_xht_row(const double* __restrict__ x, long long cs, int m, const double* sH,
                                           double (&xht)[K], double& xx) {
#pragma unroll
    for (int t = 0; t < K; t++) xht[t] = 0.0;
    xx = 0.0;
    for (int j = 0; j < m; j++) {
        const double v = x[j * cs];
        xx = fma(v, v, xx);
#pragma unroll
        for (int t = 0; t < K; t++) xht[t] = fma(v, sH[t * m + j], xht[t]);
    }
}

// The row functions read H H^T (G, K x K, shared memory) through a volatile pointer: the loads stay at their use, rather
// than being hoisted out of the row and iteration loops into K^2 registers (which spills for K >= 8).

// one coordinate-descent sweep over the K entries of a row; returns the row's share of the violation
template <int K>
__device__ __forceinline__ double fx_cd_row(double (&w)[K], const double (&xht)[K], const volatile double* G) {
    double viol = 0.0;
#pragma unroll
    for (int t = 0; t < K; t++) {
        double grad = -xht[t];
#pragma unroll
        for (int r = 0; r < K; r++) grad = fma(G[t * K + r], w[r], grad);
        viol += fabs(w[t] == 0.0 ? fmin(0.0, grad) : grad);
        const double hess = G[t * K + t];
        if (hess != 0.0) w[t] = fmax(w[t] - grad / hess, 0.0);
    }
    return viol;
}

// one multiplicative update of a row: every denominator from the row before the update
template <int K>
__device__ __forceinline__ void fx_mu_row(double (&w)[K], const double (&xht)[K], const volatile double* G) {
    double den[K];
#pragma unroll
    for (int t = 0; t < K; t++) {
        double d = 0.0;
#pragma unroll
        for (int r = 0; r < K; r++) d = fma(w[r], G[r * K + t], d);
        den[t] = d == 0.0 ? FX_MU_EPS : d;
    }
#pragma unroll
    for (int t = 0; t < K; t++) w[t] *= xht[t] / den[t];
}

// ||x_i - w_i H||^2 in the expanded form ||x_i||^2 - 2 <w_i, (X H^T)_i> + w_i (H H^T) w_i^T, which needs no X.
// Rounding: X, W, H >= 0 makes all three terms non-negative, and <W, X H^T> = <X, W H>, <W^T W, H H^T> = ||W H||^2, so
// the computed sum over all rows differs from ||X - W H||^2 by at most gamma_N ||X + W H||_F^2, gamma_N = N u / (1 - N u),
// u = 2^-53, N = m + K^2 + K + 3 + (the depth of the row reduction, <= log2(n) + 64).  The stop test compares a change
// of err against tol * err_at_init; for tol >= 1e-12 and a fit with ||X - W H|| >= 1e-3 ||X||, that bound is far below it.
template <int K>
__device__ __forceinline__ double fx_mu_row_err(const double (&w)[K], const double (&xht)[K], double xx,
                                                const volatile double* G) {
    double wx = 0.0, q = 0.0;
#pragma unroll
    for (int t = 0; t < K; t++) {
        wx = fma(w[t], xht[t], wx);
        double g = 0.0;
#pragma unroll
        for (int r = 0; r < K; r++) g = fma(G[t * K + r], w[r], g);
        q = fma(w[t], g, q);
    }
    return fma(-2.0, wx, xx) + q;
}

// ---------------------------------------------------------------------------------------------------
// resident regime
// ---------------------------------------------------------------------------------------------------
// Shared memory (doubles): sX [n][XS], sW [n][WS], sXHt [n][WS], sXX [n], sH [K][m], sHHt [K][K], sPart [2][MS_NMF_MAX_M],
// s_red [32]
template <int K>
__device__ __forceinline__ void fx_resident_body(const double* __restrict__ X, int n, int m, long long rs, long long cs,
                                                 double* __restrict__ Wp, const double* __restrict__ Hp, int solver,
                                                 int max_iter, double tol, int32_t* n_iter_out, double* err_out,
                                                 double* vaf_out, double* sm) {
    const int XS = ms_odd(m), WS = ms_odd(K);
    double* sX = sm;
    double* sW = sX + (size_t)n * XS;
    double* sXHt = sW + (size_t)n * WS;
    double* sXX = sXHt + (size_t)n * WS;
    double* sH = sXX + n;
    double* sHHt = sH + K * m;
    double* sPart = sHHt + K * K;
    double* s_red = sPart + 2 * MS_NMF_MAX_M;
    const int tid = threadIdx.x;

    for (int i = tid; i < n * m; i += FX_THREADS) sX[(i / m) * XS + i % m] = X[(i / m) * rs + (i % m) * cs];
    for (int i = tid; i < n * K; i += FX_THREADS) sW[(i / K) * WS + i % K] = Wp[i];
    for (int i = tid; i < K * m; i += FX_THREADS) sH[i] = Hp[i];
    __syncthreads();
    fx_hht<K>(sH, m, sHHt);
    for (int i = tid; i < n; i += FX_THREADS) {
        double xht[K], xx;
        fx_xht_row<K>(sX + (size_t)i * XS, 1, m, sH, xht, xx);
#pragma unroll
        for (int t = 0; t < K; t++) sXHt[i * WS + t] = xht[t];
        sXX[i] = xx;
    }
    __syncthreads();

    // the rows a thread owns are its own: only the stop tests synchronise
    const bool mu = solver == FX_SOLVER_MU, mu_checks = mu && tol > 0.0;
    double stop_ref = 0.0, prev = 0.0;  // cd: violation_init; mu: err_at_init
    if (mu_checks) {
        double e = 0.0;
        for (int i = tid; i < n; i += FX_THREADS) {
            double w[K], xht[K];
#pragma unroll
            for (int t = 0; t < K; t++) w[t] = sW[i * WS + t], xht[t] = sXHt[i * WS + t];
            e += fx_mu_row_err<K>(w, xht, sXX[i], sHHt);
        }
        stop_ref = prev = sqrt(fmax(ms_block_sum_d(e, s_red), 0.0));
    }
    int it = 0;
    for (it = 1; it <= max_iter; it++) {
        const bool check = mu ? (mu_checks && it % 10 == 0) : true;
        double part = 0.0;
        for (int i = tid; i < n; i += FX_THREADS) {
            double w[K], xht[K];
#pragma unroll
            for (int t = 0; t < K; t++) w[t] = sW[i * WS + t], xht[t] = sXHt[i * WS + t];
            if (mu) {
                fx_mu_row<K>(w, xht, sHHt);
                if (check) part += fx_mu_row_err<K>(w, xht, sXX[i], sHHt);
            } else {
                part += fx_cd_row<K>(w, xht, sHHt);
            }
#pragma unroll
            for (int t = 0; t < K; t++) sW[i * WS + t] = w[t];
        }
        if (!check) continue;
        const double total = ms_block_sum_d(part, s_red);
        if (mu) {
            const double err = sqrt(fmax(total, 0.0));
            if ((prev - err) / stop_ref < tol) break;
            prev = err;
        } else {
            if (it == 1) stop_ref = total;
            if (stop_ref == 0.0 || total / stop_ref <= tol) break;
        }
    }
    if (it > max_iter) it = max_iter;
    __syncthreads();

    // results: W, ||X - W H||_F and the variance accounted for, from X itself (one column per thread)
    for (int i = tid; i < n * K; i += FX_THREADS) Wp[i] = sW[(i / K) * WS + i % K];
    for (int j = tid; j < m; j += FX_THREADS) {
        double r2 = 0.0, c2 = 0.0;
        for (int i = 0; i < n; i++) {
            double r = sX[i * XS + j];
            c2 = fma(r, r, c2);
#pragma unroll
            for (int c = 0; c < K; c++) r = fma(-sW[i * WS + c], sH[c * m + j], r);
            r2 = fma(r, r, r2);
        }
        sPart[j] = r2;
        sPart[MS_NMF_MAX_M + j] = c2;
        vaf_out[1 + j] = 1.0 - r2 / c2;
    }
    __syncthreads();
    if (tid == 0) {
        double r2 = 0.0, c2 = 0.0;
        for (int j = 0; j < m; j++) r2 += sPart[j], c2 += sPart[MS_NMF_MAX_M + j];
        *n_iter_out = it;
        *err_out = sqrt(r2);
        vaf_out[0] = 1.0 - r2 / c2;
    }
}

__global__ void __launch_bounds__(FX_THREADS)
    ms_fx_resident_kernel(const double* __restrict__ X, int n, int m, long long rs, long long cs,
                          const MsNmfProblem* __restrict__ problems, double* __restrict__ Wg, const double* __restrict__ Hg,
                          int solver, int max_iter, double tol, int32_t* __restrict__ n_iter_out,
                          double* __restrict__ err_out, double* __restrict__ vaf_out) {
    extern __shared__ double fx_sm[];
    const MsNmfProblem pb = problems[blockIdx.x];
    const int p = blockIdx.x;
#define FX_RESIDENT(KK)                                                                                               \
    fx_resident_body<KK>(X + pb.x_off, n, m, rs, cs, Wg + pb.w_off, Hg + pb.h_off, solver, max_iter, tol,             \
                         n_iter_out + p, err_out + p, vaf_out + (long long)p * (m + 1), fx_sm)
    MS_NMF_K_SWITCH(pb.k, FX_RESIDENT)
#undef FX_RESIDENT
}

static size_t fx_resident_fixed(int m, int kmax) { return (size_t)kmax * m + (size_t)kmax * kmax + 2 * MS_NMF_MAX_M + 32; }
static size_t fx_resident_row(int m, int kmax) { return (size_t)ms_odd(m) + 2 * (size_t)ms_odd(kmax) + 1; }

// Largest n the resident fixed-H kernel takes for (m, kmax); 0 if the shape is unsupported.
extern "C" int32_t ms_nmf_fixed_h_resident_max_rows(int32_t m, int32_t kmax) {
    return ms_nmf_max_rows(m, kmax, sizeof(double), fx_resident_fixed, fx_resident_row);
}

// ---------------------------------------------------------------------------------------------------
// streaming regime
// ---------------------------------------------------------------------------------------------------
struct MsFxState {  // per problem, device memory
    double stop_ref;  // cd: violation_init; mu: err_at_init
    double prev;      // mu: the error of the previous check
    int n_iter;
    int done;
    int replay_chunk;  // 1 + the chunk in which the problem stopped (0: none) ...
    int replay_iters;  // ... after this many of its iterations
};

struct FxLayout {  // the workspace, carved by fx_layout
    MsFxState* states;  // [P]
    double* xht;        // [P][n][kmax]: X H^T rows (row stride k_p)
    double* xx;         // [P][n]: ||x_i||^2
    double* wsave;      // [P][n][kmax]: W at the start of the chunk (row stride k_p)
    double* parts;      // [P][FX_CHUNK + 1][ctas]: per-CTA sums of the stop statistic, slot s = after iteration s
    double* vparts;     // [P][vctas][2][m]: per-CTA residual / total sums of squares per column
};

static long long fx_ctas(long long n, int n_problems) {  // CTAs per problem in the streaming kernels
    long long ctas = (148LL * 8 + n_problems - 1) / n_problems, need = (n + FX_THREADS - 1) / FX_THREADS;
    return ctas < need ? ctas : need;
}
static long long fx_vaf_ctas(long long n, int m, int n_problems) {
    const int rows = FX_THREADS / m;
    long long ctas = (148LL * 8 + n_problems - 1) / n_problems, need = (n + rows - 1) / rows;
    return ctas < need ? ctas : need;
}

static size_t fx_layout(long long n, int m, int n_problems, int kmax, char* base, FxLayout* L) {
    const size_t P = (size_t)n_problems, ctas = (size_t)fx_ctas(n, n_problems), vctas = (size_t)fx_vaf_ctas(n, m, n_problems);
    size_t off = 0;
    const size_t sizes[6] = {sizeof(MsFxState) * P, sizeof(double) * P * n * kmax, sizeof(double) * P * n,
                             sizeof(double) * P * n * kmax, sizeof(double) * P * (FX_CHUNK + 1) * ctas,
                             sizeof(double) * P * vctas * 2 * m};
    void* ptrs[6];
    for (int s = 0; s < 6; s++) {
        ptrs[s] = base ? base + off : nullptr;
        off += ms_align256(sizes[s]);
    }
    if (L) {
        L->states = (MsFxState*)ptrs[0];
        L->xht = (double*)ptrs[1];
        L->xx = (double*)ptrs[2];
        L->wsave = (double*)ptrs[3];
        L->parts = (double*)ptrs[4];
        L->vparts = (double*)ptrs[5];
    }
    return off;
}

// One chunk of up to FX_CHUNK iterations for every row of one problem (grid.y).  first: form X H^T and ||x_i||^2 from
// X (the only read of X before the closing VAF pass), and for mu the error of the initial W (slot 0).
template <int K>
__device__ __forceinline__ void fx_chunk_body(const double* __restrict__ X, long long n, int m, long long rs, long long cs,
                                              double* __restrict__ Wp, const double* __restrict__ Hp, int solver, double tol,
                                              int it0, int iters, int first, double* __restrict__ xhtp,
                                              double* __restrict__ xxp, double* __restrict__ wsavep,
                                              double* __restrict__ parts, double* sm) {
    double* sH = sm;                          // [K][m]
    double* sHHt = sH + K * m;                // [K][K]
    double* sAcc = sHHt + K * K;              // [FX_CHUNK + 1][FX_THREADS]: the thread's own column
    const int tid = threadIdx.x;
    const bool mu = solver == FX_SOLVER_MU, mu_checks = mu && tol > 0.0;
    for (int i = tid; i < K * m; i += FX_THREADS) sH[i] = Hp[i];
    for (int s = 0; s <= FX_CHUNK; s++) sAcc[s * FX_THREADS + tid] = 0.0;
    __syncthreads();
    fx_hht<K>(sH, m, sHHt);
    __syncthreads();
    for (long long i = (long long)blockIdx.x * FX_THREADS + tid; i < n; i += (long long)gridDim.x * FX_THREADS) {
        double w[K], xht[K], xx;
        if (first) {
            fx_xht_row<K>(X + i * rs, cs, m, sH, xht, xx);
#pragma unroll
            for (int t = 0; t < K; t++) xhtp[i * K + t] = xht[t];
            xxp[i] = xx;
        } else {
#pragma unroll
            for (int t = 0; t < K; t++) xht[t] = xhtp[i * K + t];
            xx = xxp[i];
        }
#pragma unroll
        for (int t = 0; t < K; t++) w[t] = Wp[i * K + t], wsavep[i * K + t] = w[t];
        if (first && mu_checks) sAcc[tid] += fx_mu_row_err<K>(w, xht, xx, sHHt);
        for (int s = 1; s <= iters; s++) {
            if (mu) {
                fx_mu_row<K>(w, xht, sHHt);
                if (mu_checks && (it0 + s) % 10 == 0) sAcc[s * FX_THREADS + tid] += fx_mu_row_err<K>(w, xht, xx, sHHt);
            } else {
                sAcc[s * FX_THREADS + tid] += fx_cd_row<K>(w, xht, sHHt);
            }
        }
#pragma unroll
        for (int t = 0; t < K; t++) Wp[i * K + t] = w[t];
    }
    __syncthreads();
    for (int s = tid; s <= iters; s += FX_THREADS) {  // fixed order: thread columns 0 .. 255
        double v = 0.0;
        for (int q = 0; q < FX_THREADS; q++) v += sAcc[s * FX_THREADS + q];
        parts[(long long)s * gridDim.x + blockIdx.x] = v;
    }
}

__global__ void __launch_bounds__(FX_THREADS)
    ms_fx_chunk_kernel(const double* __restrict__ X, long long n, int m, long long rs, long long cs,
                       const MsNmfProblem* __restrict__ problems, double* __restrict__ Wg, const double* __restrict__ Hg,
                       int solver, double tol, int it0, int iters, int first, FxLayout L, int kmax) {
    extern __shared__ double fx_sm[];
    const int p = blockIdx.y;
    const MsNmfProblem pb = problems[p];
    if (L.states[p].done) return;
    double* xhtp = L.xht + (long long)p * n * kmax;
    double* wsavep = L.wsave + (long long)p * n * kmax;
    double* parts = L.parts + (long long)p * (FX_CHUNK + 1) * gridDim.x;
#define FX_CHUNK_BODY(KK)                                                                                             \
    fx_chunk_body<KK>(X + pb.x_off, n, m, rs, cs, Wg + pb.w_off, Hg + pb.h_off, solver, tol, it0, iters, first, xhtp,  \
                      L.xx + (long long)p * n, wsavep, parts, fx_sm)
    MS_NMF_K_SWITCH(pb.k, FX_CHUNK_BODY)
#undef FX_CHUNK_BODY
}

// One CTA per problem: the chunk's stop statistics, each a fixed-order sum of the CTA partials, tested iteration by
// iteration as sklearn does; the first iteration that stops the problem is recorded for the replay.
__global__ void __launch_bounds__(FX_THREADS)
    ms_fx_decide_kernel(int solver, double tol, int it0, int iters, int first, int chunk, int ctas, FxLayout L) {
    __shared__ double s_red[32];
    const int p = blockIdx.x;
    MsFxState* st = L.states + p;
    if (st->done) return;
    const double* parts = L.parts + (long long)p * (FX_CHUNK + 1) * ctas;
    const bool mu = solver == FX_SOLVER_MU, mu_checks = mu && tol > 0.0;
    double stop_ref = st->stop_ref, prev = st->prev;
    int stop = 0;
    for (int s = (first && mu_checks) ? 0 : 1; s <= iters; s++) {
        const int it = it0 + s;
        if (mu && !(mu_checks && (s == 0 || it % 10 == 0))) continue;
        double v = 0.0;
        for (int c = threadIdx.x; c < ctas; c += FX_THREADS) v += parts[(long long)s * ctas + c];
        const double total = ms_block_sum_d(v, s_red);  // the same value in every thread
        if (mu) {
            const double err = sqrt(fmax(total, 0.0));
            if (s == 0) {
                stop_ref = prev = err;
                continue;
            }
            if ((prev - err) / stop_ref < tol) {
                stop = s;
                break;
            }
            prev = err;
        } else {
            if (it == 1) stop_ref = total;
            if (stop_ref == 0.0 || total / stop_ref <= tol) {
                stop = s;
                break;
            }
        }
    }
    if (threadIdx.x == 0) {
        st->stop_ref = stop_ref;
        st->prev = prev;
        st->n_iter = it0 + (stop ? stop : iters);
        if (stop) {
            st->done = 1;
            if (stop < iters) st->replay_chunk = chunk + 1, st->replay_iters = stop;
        }
    }
}

// The rows of a problem that stopped inside chunk `chunk` run again from the chunk's saved W, up to the stop.
template <int K>
__device__ __forceinline__ void fx_replay_body(long long n, int m, double* __restrict__ Wp, const double* __restrict__ Hp,
                                               int solver, const double* __restrict__ xhtp,
                                               const double* __restrict__ wsavep, int iters, double* sm) {
    double* sH = sm;
    double* sHHt = sH + K * m;
    for (int i = threadIdx.x; i < K * m; i += FX_THREADS) sH[i] = Hp[i];
    __syncthreads();
    fx_hht<K>(sH, m, sHHt);
    __syncthreads();
    for (long long i = (long long)blockIdx.x * FX_THREADS + threadIdx.x; i < n; i += (long long)gridDim.x * FX_THREADS) {
        double w[K], xht[K];
#pragma unroll
        for (int t = 0; t < K; t++) w[t] = wsavep[i * K + t], xht[t] = xhtp[i * K + t];
        for (int s = 1; s <= iters; s++) {
            if (solver == FX_SOLVER_MU) fx_mu_row<K>(w, xht, sHHt);
            else fx_cd_row<K>(w, xht, sHHt);
        }
#pragma unroll
        for (int t = 0; t < K; t++) Wp[i * K + t] = w[t];
    }
}

__global__ void __launch_bounds__(FX_THREADS)
    ms_fx_replay_kernel(long long n, int m, const MsNmfProblem* __restrict__ problems, double* __restrict__ Wg,
                        const double* __restrict__ Hg, int solver, int chunk, FxLayout L, int kmax) {
    extern __shared__ double fx_sm[];
    const int p = blockIdx.y;
    const MsFxState st = L.states[p];
    if (st.replay_chunk != chunk + 1) return;
    const MsNmfProblem pb = problems[p];
#define FX_REPLAY(KK)                                                                                                 \
    fx_replay_body<KK>(n, m, Wg + pb.w_off, Hg + pb.h_off, solver, L.xht + (long long)p * n * kmax,                   \
                       L.wsave + (long long)p * n * kmax, st.replay_iters, fx_sm)
    MS_NMF_K_SWITCH(pb.k, FX_REPLAY)
#undef FX_REPLAY
}

// per problem (grid.y) and column: CTA sums of squares of X - W H and of X, rows of FX_THREADS / m threads in order
__global__ void __launch_bounds__(FX_THREADS)
    ms_fx_vaf_kernel(const double* __restrict__ X, long long n, int m, long long rs, long long cs,
                     const MsNmfProblem* __restrict__ problems, const double* __restrict__ Wg,
                     const double* __restrict__ Hg, FxLayout L) {
    __shared__ double sH[MS_NMF_MAX_K * MS_NMF_MAX_M];
    __shared__ double sR[2][FX_THREADS];
    const MsNmfProblem pb = problems[blockIdx.y];
    const int k = pb.k;
    const double* Xp = X + pb.x_off;
    const double* Wp = Wg + pb.w_off;
    for (int e = threadIdx.x; e < k * m; e += FX_THREADS) sH[e] = Hg[pb.h_off + e];
    __syncthreads();
    const int j = threadIdx.x % m, lane_row = threadIdx.x / m, rows_per_pass = FX_THREADS / m;
    double r2 = 0.0, c2 = 0.0;
    if (lane_row < rows_per_pass)
        for (long long i = (long long)blockIdx.x * rows_per_pass + lane_row; i < n; i += (long long)gridDim.x * rows_per_pass) {
            double r = Xp[i * rs + j * cs];
            c2 = fma(r, r, c2);
            for (int c = 0; c < k; c++) r = fma(-Wp[i * k + c], sH[c * m + j], r);
            r2 = fma(r, r, r2);
        }
    sR[0][threadIdx.x] = r2;
    sR[1][threadIdx.x] = c2;
    __syncthreads();
    if (threadIdx.x < 2 * m) {
        const int q = threadIdx.x / m, col = threadIdx.x % m;
        double v = 0.0;
        for (int l = 0; l < rows_per_pass; l++) v += sR[q][l * m + col];
        L.vparts[(((long long)blockIdx.y * gridDim.x + blockIdx.x) * 2 + q) * m + col] = v;
    }
}

__global__ void ms_fx_finish_kernel(int m, int vctas, FxLayout L, int32_t* __restrict__ n_iter, double* __restrict__ err,
                                    double* __restrict__ vaf) {
    __shared__ double s_cols[2][MS_NMF_MAX_M];
    const int p = blockIdx.x;
    const double* vp = L.vparts + (long long)p * vctas * 2 * m;
    for (int e = threadIdx.x; e < 2 * m; e += blockDim.x) {
        double v = 0.0;
        for (int c = 0; c < vctas; c++) v += vp[(long long)c * 2 * m + e];
        s_cols[e / m][e % m] = v;
    }
    __syncthreads();
    for (int j = threadIdx.x; j < m; j += blockDim.x) vaf[(long long)p * (m + 1) + 1 + j] = 1.0 - s_cols[0][j] / s_cols[1][j];
    if (threadIdx.x == 0) {
        double r2 = 0.0, c2 = 0.0;
        for (int j = 0; j < m; j++) r2 += s_cols[0][j], c2 += s_cols[1][j];
        vaf[(long long)p * (m + 1)] = 1.0 - r2 / c2;
        err[p] = sqrt(r2);
        n_iter[p] = L.states[p].n_iter;
    }
}

// ---------------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------------
extern "C" int64_t ms_nmf_fixed_h_workspace_bytes(int64_t n, int32_t m, int32_t n_problems, int32_t kmax) {
    if (n < 1 || m < 1 || m > MS_NMF_MAX_M || n_problems < 0 || kmax < 1 || kmax > MS_NMF_MAX_K) return 0;
    if (n_problems == 0) return 256;
    return (int64_t)fx_layout(n, m, n_problems, kmax, nullptr, nullptr) + 256;
}

extern "C" int ms_nmf_fixed_h(const double* d_X, int64_t n, int32_t m, int64_t row_stride, int64_t col_stride,
                              const void* d_table, int32_t n_problems, int32_t kmax, double* d_W, const double* d_H,
                              int32_t solver, int32_t max_iter, double tol, int32_t regime, void* d_work,
                              int32_t* d_n_iter, double* d_err, double* d_vaf, void* stream) {
    if (!d_X || !d_table || !d_W || !d_H || !d_n_iter || !d_err || !d_vaf) return MS_E_INVALID;
    if (n < 1 || m < 1 || m > MS_NMF_MAX_M || kmax < 1 || kmax > MS_NMF_MAX_K || n_problems < 0 || max_iter < 0 ||
        !(tol >= 0.0) || (solver != FX_SOLVER_CD && solver != FX_SOLVER_MU) || (regime != 0 && regime != 1) ||
        row_stride < 0 || col_stride < 0)
        return MS_E_INVALID;
    if (n_problems == 0) return MS_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const MsNmfProblem* d_problems = (const MsNmfProblem*)d_table;
    if (regime == 0) {
        if (n > ms_nmf_fixed_h_resident_max_rows(m, kmax)) return MS_E_INVALID;  // too long for shared memory
        const size_t smem = sizeof(double) * ((size_t)n * fx_resident_row(m, kmax) + fx_resident_fixed(m, kmax));
        MS_CUDA_CHECK(cudaFuncSetAttribute(ms_fx_resident_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ms_fx_resident_kernel<<<n_problems, FX_THREADS, smem, st>>>(d_X, (int)n, m, row_stride, col_stride, d_problems, d_W,
                                                                    d_H, solver, max_iter, tol, d_n_iter, d_err, d_vaf);
        MS_COUNT_LAUNCH();
        MS_CUDA_CHECK(cudaGetLastError());
        return MS_OK;
    }
    if (!d_work) return MS_E_INVALID;
    FxLayout L;
    fx_layout(n, m, n_problems, kmax, (char*)d_work, &L);
    const int ctas = (int)fx_ctas(n, n_problems), vctas = (int)fx_vaf_ctas(n, m, n_problems);
    MS_CUDA_CHECK(cudaMemsetAsync(L.states, 0, sizeof(MsFxState) * (size_t)n_problems, st));
    const size_t smem_chunk = sizeof(double) * ((size_t)kmax * MS_NMF_MAX_M + kmax * kmax + (FX_CHUNK + 1) * FX_THREADS);
    const size_t smem_replay = sizeof(double) * ((size_t)kmax * MS_NMF_MAX_M + kmax * kmax);
    MS_CUDA_CHECK(cudaFuncSetAttribute(ms_fx_chunk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_chunk));
    for (int it0 = 0, chunk = 0; it0 < max_iter || chunk == 0; it0 += FX_CHUNK, chunk++) {
        const int iters = max_iter - it0 < FX_CHUNK ? max_iter - it0 : FX_CHUNK;
        const int first = chunk == 0;
        ms_fx_chunk_kernel<<<dim3(ctas, n_problems), FX_THREADS, smem_chunk, st>>>(
            d_X, n, m, row_stride, col_stride, d_problems, d_W, d_H, solver, tol, it0, iters, first, L, kmax);
        MS_COUNT_LAUNCH();
        ms_fx_decide_kernel<<<n_problems, FX_THREADS, 0, st>>>(solver, tol, it0, iters, first, chunk, ctas, L);
        MS_COUNT_LAUNCH();
        ms_fx_replay_kernel<<<dim3(ctas, n_problems), FX_THREADS, smem_replay, st>>>(n, m, d_problems, d_W, d_H, solver,
                                                                                     chunk, L, kmax);
        MS_COUNT_LAUNCH();
        if (chunk % 2 == 1 && it0 + iters < max_iter) {  // stop early once every problem is done
            const int done = ms_nmf_all_done(L.states, n_problems, st);
            if (done < 0) return done;
            if (done) break;
        }
    }
    ms_fx_vaf_kernel<<<dim3(vctas, n_problems), FX_THREADS, 0, st>>>(d_X, n, m, row_stride, col_stride, d_problems, d_W,
                                                                     d_H, L);
    MS_COUNT_LAUNCH();
    ms_fx_finish_kernel<<<n_problems, 64, 0, st>>>(m, vctas, L, d_n_iter, d_err, d_vaf);
    MS_COUNT_LAUNCH();
    MS_CUDA_CHECK(cudaGetLastError());
    return MS_OK;
}
