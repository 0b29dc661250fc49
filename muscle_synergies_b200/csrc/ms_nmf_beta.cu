// β-divergence NMF by multiplicative updates (beta_loss != 2), fp64: fit (W and H) and transform (H fixed).
//
// scikit-learn 1.9.0's _fit_multiplicative_update (sklearn/decomposition/_nmf.py), dense X, no regularisation, with
// EPSILON = float32 eps and gamma = 1 / (2 - beta) (beta < 1), 1 / (beta - 1) (beta > 2), 1 otherwise:
//
//   W step (WH from the old W):  W *= ((X * WHs^(beta-2)) H^T / D)^gamma,  D = rowsum(H) (KL) or WHd^(beta-1) H^T
//   H step (WH from the new W):  H *= (W^T (X * WHs^(beta-2)) / D)^gamma,  D = colsum(W), 0 -> 1 (KL) or W^T WHd^(beta-1)
//     WHs = WH clamped below at EPSILON for beta < 2, WHd = WH clamped for beta < 1; a zero D becomes EPSILON;
//     after the W step W < float64 eps -> 0 for beta < 1, after the H step H < eps -> 0 for beta <= 1
//   stop (tol > 0, every 10 iterations): err = sqrt(2 max(D_beta(X | W H), 0)), stop when (prev - err) / err_init < tol
//
// Powers follow numpy's scalar fast paths (x^2 = x * x, x^1 = x, x^0.5 = sqrt, x^-1 = 1 / x), so KL (beta = 1) and
// Itakura-Saito (beta = 0) never call pow; KL and IS are compile-time specialisations, every other beta the general one.
// D_beta is summed element by element (each element's terms together) rather than as sklearn's separate sums: the same
// value up to rounding.
//
// Unlike the Frobenius kernels there is no Gram-matrix shortcut: every update and every stop test needs WH element by
// element.  One thread owns a row of W; the row function bt_row computes the row's WH twice (old W for its own update,
// new W for the H-step terms X * WHs^(beta-2) and WHd^(beta-1), which it leaves in shared memory), and bt_hacc sums
// those terms over rows, one (t, j) entry of H per thread.
//
//   ms_bt_resident_kernel   one CTA per problem: X, W, H and the H-step terms in shared memory
//   ms_bt_pass_kernel       long signals, one launch per iteration: rows in tiles, the W step of a row and that row's
//   ms_bt_update_kernel     H-step terms in one pass over X; per-CTA partial sums to the workspace; then one CTA per
//                           problem sums them in a fixed order and applies the H update.  The divergence a stop test
//                           needs rides along with the next pass (its W step computes the WH of the tested W and H); a
//                           problem that stops gets back the W that pass saved and keeps its H, so n_iter, W and H are
//                           those of the iteration sklearn stops at
//   ms_bt_final_kernel      the final divergence (err) and ||X - W H|| per column (VAF), CTA partials, then
//   ms_bt_finish_kernel     summed in a fixed order
//
// No floating-point atomics: two identical calls give bit-identical W, H, n_iter, err and VAF.  The two regimes sum the
// H-step terms in different orders, so they agree to rounding, not bit for bit.
#include <stdio.h>

#include "ms_common.cuh"

#define BT_THREADS 256
#define BT_MAX_K 16
#define BT_MAX_M 64
#define BT_EPS 1.1920928955078125e-07        // np.finfo(np.float32).eps, sklearn's EPSILON
#define BT_DBL_EPS 2.220446049250313e-16     // np.finfo(np.float64).eps
#define BT_IS 0
#define BT_KL 1
#define BT_GEN 2
#define BT_Q(K) (((K) * BT_MAX_M + BT_THREADS - 1) / BT_THREADS)  // H entries per thread in bt_hacc

struct MsNmfProblem {  // ms_nmf_plan's table (csrc/ms_nmf.cu)
    int k;
    long long w_off;
    long long h_off;
    long long x_off;
};

__host__ __device__ inline int bt_odd(int v) { return v | 1; }

// numpy's x ** e for a scalar e: the fast paths first, pow otherwise
__device__ __forceinline__ double bt_pow(double x, double e) {
    if (e == 2.0) return x * x;
    if (e == 1.0) return x;
    if (e == 0.5) return sqrt(x);
    if (e == -1.0) return 1.0 / x;
    if (e == 0.0) return 1.0;
    return pow(x, e);
}

__device__ __forceinline__ double bt_clamp(double wh) { return wh < BT_EPS ? BT_EPS : wh; }

// the H-step / W-step terms of one element: f = X * WHs^(beta-2), g = WHd^(beta-1) (unused for KL)
template <int MODE>
__device__ __forceinline__ void bt_fg(double x, double wh, double beta, double& f, double& g) {
    if (MODE == BT_KL) {
        f = x / bt_clamp(wh);
        g = 0.0;
    } else if (MODE == BT_IS) {
        const double r = 1.0 / bt_clamp(wh);  // (WH^-1)^2 * X, and WH^-1
        f = r * r * x;
        g = r;
    } else {
        f = bt_pow(beta < 2.0 ? bt_clamp(wh) : wh, beta - 2.0) * x;
        g = bt_pow(beta < 1.0 ? bt_clamp(wh) : wh, beta - 1.0);
    }
}

// one element's share of D_beta(X | WH) (before the general case's 1 / (beta (beta - 1))); X <= EPSILON drops the X terms
template <int MODE>
__device__ __forceinline__ double bt_div_term(double x, double wh, double beta) {
    if (MODE == BT_KL) {
        double t = wh;
        if (x > BT_EPS) t += x * log(x / bt_clamp(wh)) - x;
        return t;
    } else if (MODE == BT_IS) {
        if (!(x > BT_EPS)) return -1.0;
        const double d = x / bt_clamp(wh);
        return d - log(d) - 1.0;
    } else {
        double t = (beta - 1.0) * bt_pow(wh, beta);
        if (x > BT_EPS) t += bt_pow(x, beta) - beta * (x * bt_pow(bt_clamp(wh), beta - 1.0));
        return t;
    }
}

// err = sqrt(2 max(res, 0)) of a summed divergence (a NaN stays NaN, as in Python's max)
__device__ __forceinline__ double bt_err(int mode, double total, double beta) {
    double res = mode == BT_GEN ? total / (beta * (beta - 1.0)) : total;
    if (res < 0.0) res = 0.0;
    return sqrt(2.0 * res);
}

// the update ratio to the power gamma: 1 for KL, 1/2 (numpy's sqrt) for IS, at run time for the general case
template <int MODE>
__device__ __forceinline__ double bt_gamma(double r, double gamma) {
    if (MODE == BT_KL) return r;
    if (MODE == BT_IS) return sqrt(r);
    return gamma == 1.0 ? r : bt_pow(r, gamma);
}

// one H entry's update from its summed numerator and denominator
template <int MODE>
__device__ __forceinline__ double bt_h_update(double h, double num, double den, double beta, double gamma) {
    if (MODE == BT_KL && den == 0.0) den = 1.0;
    if (den == 0.0) den = BT_EPS;
    h *= bt_gamma<MODE>(num / den, gamma);
    if (beta <= 1.0 && h < BT_DBL_EPS) h = 0.0;
    return h;
}

// The W step of one row (X element j at x[j * cs]; sH [K][m], sHs = rowsum(H) for KL).  do_div adds the divergence of the
// row's current W and H to div.  sF != nullptr: leaves the H-step terms of the updated row in sF[j], sG[j].
template <int MODE, int K>
__device__ __forceinline__ void bt_row(double (&w)[K], const double* __restrict__ x, long long cs, int m, const double* sH,
                                       const double* sHs, double beta, double gamma, bool do_div, double& div,
                                       double* sF, double* sG) {
    double num[K], den[K];
#pragma unroll
    for (int t = 0; t < K; t++) num[t] = 0.0, den[t] = 0.0;
    for (int j = 0; j < m; j++) {
        double wh = 0.0;
#pragma unroll
        for (int t = 0; t < K; t++) wh = fma(w[t], sH[t * m + j], wh);
        const double xv = x[j * cs];
        if (do_div) div += bt_div_term<MODE>(xv, wh, beta);
        double f, g;
        bt_fg<MODE>(xv, wh, beta, f, g);
#pragma unroll
        for (int t = 0; t < K; t++) {
            num[t] = fma(f, sH[t * m + j], num[t]);
            if (MODE != BT_KL) den[t] = fma(g, sH[t * m + j], den[t]);
        }
    }
#pragma unroll
    for (int t = 0; t < K; t++) {
        double d = MODE == BT_KL ? sHs[t] : den[t];
        if (d == 0.0) d = BT_EPS;
        w[t] *= bt_gamma<MODE>(num[t] / d, gamma);
        if (beta < 1.0 && w[t] < BT_DBL_EPS) w[t] = 0.0;
    }
    if (sF) {
        for (int j = 0; j < m; j++) {
            double wh = 0.0;
#pragma unroll
            for (int t = 0; t < K; t++) wh = fma(w[t], sH[t * m + j], wh);
            double f, g;
            bt_fg<MODE>(x[j * cs], wh, beta, f, g);
            sF[j] = f;
            if (MODE != BT_KL) sG[j] = g;
        }
    }
}

// the divergence of `rows` rows (W rows in sW, row stride WS) with the current H, this thread's rows only
template <int MODE, int K>
__device__ __forceinline__ double bt_div_rows(const double* sX, int XS, const double* sW, int WS, int rows, int m,
                                              const double* sH, double beta) {
    double div = 0.0;
    for (int i = threadIdx.x; i < rows; i += BT_THREADS)
        for (int j = 0; j < m; j++) {
            double wh = 0.0;
#pragma unroll
            for (int t = 0; t < K; t++) wh = fma(sW[i * WS + t], sH[t * m + j], wh);
            div += bt_div_term<MODE>(sX[i * XS + j], wh, beta);
        }
    return div;
}

// H-step sums over `rows` rows, one (t, j) entry per thread (q-th: e = tid + q * BT_THREADS), rows in order:
// an += W[r][t] F[r][j], ad += W[r][t] G[r][j] (KL: ad += W[r][t], the column sum of W)
template <int MODE, int K>
__device__ __forceinline__ void bt_hacc(const double* sW, int WS, const double* sF, const double* sG, int XS, int rows,
                                        int m, double (&an)[BT_Q(K)], double (&ad)[BT_Q(K)]) {
#pragma unroll
    for (int q = 0; q < BT_Q(K); q++) {
        const int e = threadIdx.x + q * BT_THREADS;
        if (e >= K * m) break;
        const int t = e / m, j = e % m;
        double a = an[q], d = ad[q];
        for (int r = 0; r < rows; r++) {
            const double wt = sW[r * WS + t];
            a = fma(wt, sF[r * XS + j], a);
            d = MODE == BT_KL ? d + wt : fma(wt, sG[r * XS + j], d);
        }
        an[q] = a, ad[q] = d;
    }
}

// rowsum(H) for KL's W step
__device__ __forceinline__ void bt_hsum(const double* sH, int k, int m, double* sHs) {
    for (int t = threadIdx.x; t < k; t += BT_THREADS) {
        double s = 0.0;
        for (int j = 0; j < m; j++) s += sH[t * m + j];
        sHs[t] = s;
    }
}

// fixed-order sum over the CTA (warp trees, then the warps in order); every thread gets the total
__device__ __forceinline__ double bt_block_sum(double v, double* s_red) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    double total = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) total += s_red[w];
    return total;
}

#define BT_K_SWITCH(KEXPR, CALL)                                                                                      \
    switch (KEXPR) {                                                                                                  \
        case 1: CALL(1); break;   case 2: CALL(2); break;   case 3: CALL(3); break;   case 4: CALL(4); break;         \
        case 5: CALL(5); break;   case 6: CALL(6); break;   case 7: CALL(7); break;   case 8: CALL(8); break;         \
        case 9: CALL(9); break;   case 10: CALL(10); break; case 11: CALL(11); break; case 12: CALL(12); break;       \
        case 13: CALL(13); break; case 14: CALL(14); break; case 15: CALL(15); break; case 16: CALL(16); break;       \
        default: break;                                                                                               \
    }

// ---------------------------------------------------------------------------------------------------
// resident regime
// ---------------------------------------------------------------------------------------------------
// Shared memory (doubles): sX [n][XS], sF [n][XS], sG [n][XS], sW [n][WS], sH [K][m], sHs [K], sPart [2][BT_MAX_M],
// s_red [32]
template <int MODE, int K>
__device__ __forceinline__ void bt_resident_body(const double* __restrict__ X, int n, int m, long long rs, long long cs,
                                                 double* __restrict__ Wp, double* __restrict__ Hp, double beta,
                                                 double gamma, int update_H, int max_iter, double tol,
                                                 int32_t* n_iter_out, double* err_out, double* vaf_out, double* sm) {
    const int XS = bt_odd(m), WS = bt_odd(K);
    double* sX = sm;
    double* sF = sX + (size_t)n * XS;
    double* sG = sF + (size_t)n * XS;
    double* sW = sG + (size_t)n * XS;
    double* sH = sW + (size_t)n * WS;
    double* sHs = sH + K * m;
    double* sPart = sHs + K;
    double* s_red = sPart + 2 * BT_MAX_M;
    const int tid = threadIdx.x;

    for (int i = tid; i < n * m; i += BT_THREADS) sX[(i / m) * XS + i % m] = X[(i / m) * rs + (i % m) * cs];
    for (int i = tid; i < n * K; i += BT_THREADS) sW[(i / K) * WS + i % K] = Wp[i];
    for (int i = tid; i < K * m; i += BT_THREADS) sH[i] = Hp[i];
    __syncthreads();
    if (MODE == BT_KL) bt_hsum(sH, K, m, sHs);
    __syncthreads();

    double stop_ref = 0.0, prev = 0.0, unused = 0.0;
    if (tol > 0.0) stop_ref = prev = bt_err(MODE, bt_block_sum(bt_div_rows<MODE, K>(sX, XS, sW, WS, n, m, sH, beta), s_red), beta);
    int it = 0;
    for (it = 1; it <= max_iter; it++) {
        for (int i = tid; i < n; i += BT_THREADS) {
            double w[K];
#pragma unroll
            for (int t = 0; t < K; t++) w[t] = sW[i * WS + t];
            bt_row<MODE, K>(w, sX + (size_t)i * XS, 1, m, sH, sHs, beta, gamma, false, unused,
                            update_H ? sF + (size_t)i * XS : nullptr, sG + (size_t)i * XS);
#pragma unroll
            for (int t = 0; t < K; t++) sW[i * WS + t] = w[t];
        }
        if (update_H) {
            __syncthreads();  // every row's W and H-step terms are in place; nobody reads sH until the next barrier
            double an[BT_Q(K)], ad[BT_Q(K)];
#pragma unroll
            for (int q = 0; q < BT_Q(K); q++) an[q] = 0.0, ad[q] = 0.0;
            bt_hacc<MODE, K>(sW, WS, sF, sG, XS, n, m, an, ad);
#pragma unroll
            for (int q = 0; q < BT_Q(K); q++) {
                const int e = tid + q * BT_THREADS;
                if (e < K * m) sH[e] = bt_h_update<MODE>(sH[e], an[q], ad[q], beta, gamma);
            }
            __syncthreads();
            if (MODE == BT_KL) {
                bt_hsum(sH, K, m, sHs);
                __syncthreads();
            }
        }
        if (tol > 0.0 && it % 10 == 0) {
            const double err =
                bt_err(MODE, bt_block_sum(bt_div_rows<MODE, K>(sX, XS, sW, WS, n, m, sH, beta), s_red), beta);
            if ((prev - err) / stop_ref < tol) break;
            prev = err;
        }
    }
    if (it > max_iter) it = max_iter;
    __syncthreads();

    // results: W, H, the divergence (sklearn's reconstruction_err_) and the Frobenius VAF, from X itself
    for (int i = tid; i < n * K; i += BT_THREADS) Wp[i] = sW[(i / K) * WS + i % K];
    if (update_H)
        for (int i = tid; i < K * m; i += BT_THREADS) Hp[i] = sH[i];
    const double err = bt_err(MODE, bt_block_sum(bt_div_rows<MODE, K>(sX, XS, sW, WS, n, m, sH, beta), s_red), beta);
    for (int j = tid; j < m; j += BT_THREADS) {
        double r2 = 0.0, c2 = 0.0;
        for (int i = 0; i < n; i++) {
            double r = sX[i * XS + j];
            c2 = fma(r, r, c2);
#pragma unroll
            for (int c = 0; c < K; c++) r = fma(-sW[i * WS + c], sH[c * m + j], r);
            r2 = fma(r, r, r2);
        }
        sPart[j] = r2;
        sPart[BT_MAX_M + j] = c2;
        vaf_out[1 + j] = 1.0 - r2 / c2;
    }
    __syncthreads();
    if (tid == 0) {
        double r2 = 0.0, c2 = 0.0;
        for (int j = 0; j < m; j++) r2 += sPart[j], c2 += sPart[BT_MAX_M + j];
        *n_iter_out = it;
        *err_out = err;
        vaf_out[0] = 1.0 - r2 / c2;
    }
}

// __maxnreg__ rather than __launch_bounds__: ptxas otherwise holds the KL specialisation to 128 registers and spills
template <int MODE>
__global__ void __maxnreg__(255)
    ms_bt_resident_kernel(const double* __restrict__ X, int n, int m, long long rs, long long cs,
                          const MsNmfProblem* __restrict__ problems, double* __restrict__ Wg, double* __restrict__ Hg,
                          double beta, double gamma, int update_H, int max_iter, double tol,
                          int32_t* __restrict__ n_iter_out, double* __restrict__ err_out, double* __restrict__ vaf_out) {
    extern __shared__ double bt_sm[];
    const MsNmfProblem pb = problems[blockIdx.x];
    const int p = blockIdx.x;
#define BT_RESIDENT(KK)                                                                                               \
    bt_resident_body<MODE, KK>(X + pb.x_off, n, m, rs, cs, Wg + pb.w_off, Hg + pb.h_off, beta, gamma, update_H,       \
                               max_iter, tol, n_iter_out + p, err_out + p, vaf_out + (long long)p * (m + 1), bt_sm)
    BT_K_SWITCH(pb.k, BT_RESIDENT)
#undef BT_RESIDENT
}

static size_t bt_resident_fixed(int m, int kmax) { return (size_t)kmax * m + kmax + 2 * BT_MAX_M + 32; }
static size_t bt_resident_row(int m, int kmax) { return 3 * (size_t)bt_odd(m) + bt_odd(kmax); }
static const size_t BT_SMEM_BUDGET = 227 * 1024 - 1024;

// Largest n the resident β kernel takes for (m, kmax); 0 if the shape is unsupported.
extern "C" int32_t ms_nmf_beta_resident_max_rows(int32_t m, int32_t kmax) {
    if (m < 1 || m > BT_MAX_M || kmax < 1 || kmax > BT_MAX_K) return 0;
    return (int32_t)((BT_SMEM_BUDGET - sizeof(double) * bt_resident_fixed(m, kmax)) /
                     (sizeof(double) * bt_resident_row(m, kmax)));
}

// ---------------------------------------------------------------------------------------------------
// streaming regime
// ---------------------------------------------------------------------------------------------------
struct MsBtState {  // per problem, device memory
    double stop_ref;  // err_at_init
    double prev;      // the error of the previous check
    int n_iter;
    int done;
    int pending;  // the iteration whose divergence the next pass computes (0: the init), -1: none
    int restore;  // stopped at `pending`: W comes back from wsave
};

struct BtLayout {  // the workspace, carved by bt_layout
    MsBtState* states;  // [P]
    double* wsave;      // [P][n][kmax]: W of the iteration under test (row stride k_p)
    double* parts;      // [P][ctas][2 kmax m + 1]: per-CTA H-step numerators, denominators, then the divergence
    double* vparts;     // [P][vctas][2 m + 1]: per-CTA residual / total sums of squares per column, then the divergence
};

static size_t bt_align(size_t b) { return (b + 255) / 256 * 256; }

// rows per tile of the pass kernel: one per thread, fewer where the H-step terms of 256 rows do not fit
static int bt_tile_rows(int m, int kmax) {
    const size_t fixed = (size_t)kmax * m + kmax + 32, row = 2 * (size_t)bt_odd(m) + bt_odd(kmax);
    const size_t fit = (BT_SMEM_BUDGET / sizeof(double) - fixed) / row;
    return (int)(fit < BT_THREADS ? fit : BT_THREADS);
}
static size_t bt_pass_smem(int m, int kmax) {
    return sizeof(double) * ((size_t)kmax * m + kmax + 32 +
                             (size_t)bt_tile_rows(m, kmax) * (2 * (size_t)bt_odd(m) + bt_odd(kmax)));
}
static long long bt_ctas(long long n, int m, int kmax, int n_problems) {  // pass-kernel CTAs per problem
    const long long tr = bt_tile_rows(m, kmax);
    long long ctas = (148LL * 2 + n_problems - 1) / n_problems, need = (n + tr - 1) / tr;
    return ctas < need ? ctas : need;
}
static long long bt_vaf_ctas(long long n, int m, int n_problems) {
    const int rows = BT_THREADS / m;
    long long ctas = (148LL * 8 + n_problems - 1) / n_problems, need = (n + rows - 1) / rows;
    return ctas < need ? ctas : need;
}
__host__ __device__ inline size_t bt_part_stride(int m, int kmax) { return 2 * (size_t)kmax * m + 1; }

static size_t bt_layout(long long n, int m, int n_problems, int kmax, char* base, BtLayout* L) {
    const size_t P = (size_t)n_problems, ctas = (size_t)bt_ctas(n, m, kmax, n_problems),
                 vctas = (size_t)bt_vaf_ctas(n, m, n_problems);
    const size_t sizes[4] = {sizeof(MsBtState) * P, sizeof(double) * P * n * kmax,
                             sizeof(double) * P * ctas * bt_part_stride(m, kmax), sizeof(double) * P * vctas * (2 * m + 1)};
    void* ptrs[4];
    size_t off = 0;
    for (int s = 0; s < 4; s++) {
        ptrs[s] = base ? base + off : nullptr;
        off += bt_align(sizes[s]);
    }
    if (L) {
        L->states = (MsBtState*)ptrs[0];
        L->wsave = (double*)ptrs[1];
        L->parts = (double*)ptrs[2];
        L->vparts = (double*)ptrs[3];
    }
    return off;
}

__global__ void ms_bt_init_kernel(int n_problems, int max_iter, double tol, BtLayout L) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_problems) return;
    MsBtState s;
    s.stop_ref = s.prev = 0.0;
    s.n_iter = 0;
    s.done = max_iter == 0;
    s.pending = tol > 0.0 ? 0 : -1;
    s.restore = 0;
    L.states[p] = s;
}

// One iteration's pass over one problem's rows (grid.y = problem), tiles of TR rows: the W step of each row (and, when a
// stop test is pending, the divergence of the W and H under test, with that W saved), then the tile's H-step sums.
template <int MODE, int K>
__device__ __forceinline__ void bt_pass_body(const double* __restrict__ X, long long n, int m, long long rs, long long cs,
                                             double* __restrict__ Wp, const double* __restrict__ Hp, double beta,
                                             double gamma, int update_H, bool do_div, int TR,
                                             double* __restrict__ wsavep, double* __restrict__ part, double* sm) {
    const int XS = bt_odd(m), WS = bt_odd(K);
    double* sH = sm;
    double* sHs = sH + K * m;
    double* s_red = sHs + K;
    double* sW = s_red + 32;
    double* sF = sW + (size_t)TR * WS;
    double* sG = sF + (size_t)TR * XS;
    const int tid = threadIdx.x;
    for (int i = tid; i < K * m; i += BT_THREADS) sH[i] = Hp[i];
    __syncthreads();
    if (MODE == BT_KL) bt_hsum(sH, K, m, sHs);
    __syncthreads();
    double an[BT_Q(K)], ad[BT_Q(K)], div = 0.0;
#pragma unroll
    for (int q = 0; q < BT_Q(K); q++) an[q] = 0.0, ad[q] = 0.0;
    for (long long r0 = (long long)blockIdx.x * TR; r0 < n; r0 += (long long)gridDim.x * TR) {
        const int rows = n - r0 < TR ? (int)(n - r0) : TR;
        if (tid < rows) {
            const long long i = r0 + tid;
            double w[K];
#pragma unroll
            for (int t = 0; t < K; t++) w[t] = Wp[i * K + t];
            if (do_div) {
#pragma unroll
                for (int t = 0; t < K; t++) wsavep[i * K + t] = w[t];
            }
            bt_row<MODE, K>(w, X + i * rs, cs, m, sH, sHs, beta, gamma, do_div, div,
                            update_H ? sF + (size_t)tid * XS : nullptr, sG + (size_t)tid * XS);
#pragma unroll
            for (int t = 0; t < K; t++) Wp[i * K + t] = w[t], sW[tid * WS + t] = w[t];
        }
        if (update_H) {
            __syncthreads();
            bt_hacc<MODE, K>(sW, WS, sF, sG, XS, rows, m, an, ad);
            __syncthreads();
        }
    }
    if (update_H) {
#pragma unroll
        for (int q = 0; q < BT_Q(K); q++) {
            const int e = tid + q * BT_THREADS;
            if (e < K * m) part[e] = an[q], part[K * m + e] = ad[q];
        }
    }
    if (do_div) {
        const double total = bt_block_sum(div, s_red);
        if (tid == 0) part[2 * K * m] = total;
    }
}

template <int MODE>
__global__ void __launch_bounds__(BT_THREADS)
    ms_bt_pass_kernel(const double* __restrict__ X, long long n, int m, long long rs, long long cs,
                      const MsNmfProblem* __restrict__ problems, double* __restrict__ Wg, const double* __restrict__ Hg,
                      double beta, double gamma, int update_H, int TR, BtLayout L, int kmax) {
    extern __shared__ double bt_sm[];
    const int p = blockIdx.y;
    const MsBtState st = L.states[p];
    if (st.done) return;
    const MsNmfProblem pb = problems[p];
    double* part = L.parts + ((long long)p * gridDim.x + blockIdx.x) * bt_part_stride(m, kmax);
#define BT_PASS(KK)                                                                                                   \
    bt_pass_body<MODE, KK>(X + pb.x_off, n, m, rs, cs, Wg + pb.w_off, Hg + pb.h_off, beta, gamma, update_H,           \
                           st.pending >= 0, TR, L.wsave + (long long)p * n * kmax, part, bt_sm)
    BT_K_SWITCH(pb.k, BT_PASS)
#undef BT_PASS
}

// One CTA per problem after the pass of iteration `it`: the pending stop test (CTA partials summed in order), then the
// H update from the CTA partials, each entry summed in CTA order.
__global__ void __launch_bounds__(BT_THREADS)
    ms_bt_update_kernel(const MsNmfProblem* __restrict__ problems, double* __restrict__ Hg, int m, int mode, double beta,
                        double gamma, int update_H, int it, int max_iter, double tol, int ctas, BtLayout L, int kmax) {
    __shared__ int s_stop;
    const int p = blockIdx.x;
    MsBtState st = L.states[p];
    if (st.done) return;
    const int k = problems[p].k;
    const size_t PS = bt_part_stride(m, kmax);
    const double* parts = L.parts + (long long)p * ctas * PS;
    if (threadIdx.x == 0) {
        int stop = 0;
        if (st.pending >= 0) {
            double total = 0.0;
            for (int c = 0; c < ctas; c++) total += parts[c * PS + 2 * k * m];
            const double err = bt_err(mode, total, beta);
            if (st.pending == 0) {
                st.stop_ref = st.prev = err;
            } else if ((st.prev - err) / st.stop_ref < tol) {
                stop = 1;
                st.done = 1;
                st.restore = 1;
                st.n_iter = st.pending;
            } else {
                st.prev = err;
            }
        }
        if (!stop) {
            st.n_iter = it;
            st.pending = (tol > 0.0 && it % 10 == 0 && it < max_iter) ? it : -1;
            st.done = it >= max_iter;
        }
        L.states[p] = st;
        s_stop = stop;
    }
    __syncthreads();
    if (s_stop || !update_H) return;
    double* Hp = Hg + problems[p].h_off;
    for (int e = threadIdx.x; e < k * m; e += BT_THREADS) {
        double num = 0.0, den = 0.0;
        for (int c = 0; c < ctas; c++) num += parts[c * PS + e], den += parts[c * PS + k * m + e];
        Hp[e] = mode == BT_KL   ? bt_h_update<BT_KL>(Hp[e], num, den, beta, gamma)
                : mode == BT_IS ? bt_h_update<BT_IS>(Hp[e], num, den, beta, gamma)
                                : bt_h_update<BT_GEN>(Hp[e], num, den, beta, gamma);
    }
}

// a problem that stopped at the iteration under test takes back that iteration's W
__global__ void __launch_bounds__(BT_THREADS)
    ms_bt_restore_kernel(long long n, const MsNmfProblem* __restrict__ problems, double* __restrict__ Wg, BtLayout L,
                         int kmax) {
    const int p = blockIdx.y;
    if (!L.states[p].restore) return;
    const MsNmfProblem pb = problems[p];
    const double* ws = L.wsave + (long long)p * n * kmax;
    for (long long e = (long long)blockIdx.x * BT_THREADS + threadIdx.x; e < n * pb.k; e += (long long)gridDim.x * BT_THREADS)
        Wg[pb.w_off + e] = ws[e];
}

// per problem (grid.y) and column: CTA sums of squares of X - W H and of X, rows of BT_THREADS / m threads in order,
// and the CTA's divergence
template <int MODE>
__global__ void __launch_bounds__(BT_THREADS)
    ms_bt_final_kernel(const double* __restrict__ X, long long n, int m, long long rs, long long cs,
                       const MsNmfProblem* __restrict__ problems, const double* __restrict__ Wg,
                       const double* __restrict__ Hg, double beta, BtLayout L) {
    __shared__ double sH[BT_MAX_K * BT_MAX_M];
    __shared__ double sR[3][BT_THREADS];
    const MsNmfProblem pb = problems[blockIdx.y];
    const int k = pb.k;
    const double* Xp = X + pb.x_off;
    const double* Wp = Wg + pb.w_off;
    for (int e = threadIdx.x; e < k * m; e += BT_THREADS) sH[e] = Hg[pb.h_off + e];
    __syncthreads();
    const int j = threadIdx.x % m, lane_row = threadIdx.x / m, rows_per_pass = BT_THREADS / m;
    double r2 = 0.0, c2 = 0.0, div = 0.0;
    if (lane_row < rows_per_pass)
        for (long long i = (long long)blockIdx.x * rows_per_pass + lane_row; i < n; i += (long long)gridDim.x * rows_per_pass) {
            const double x = Xp[i * rs + j * cs];
            double wh = 0.0;
            for (int c = 0; c < k; c++) wh = fma(Wp[i * k + c], sH[c * m + j], wh);
            div += bt_div_term<MODE>(x, wh, beta);
            double r = x;
            c2 = fma(r, r, c2);
            for (int c = 0; c < k; c++) r = fma(-Wp[i * k + c], sH[c * m + j], r);
            r2 = fma(r, r, r2);
        }
    sR[0][threadIdx.x] = r2;
    sR[1][threadIdx.x] = c2;
    sR[2][threadIdx.x] = div;
    __syncthreads();
    double* vp = L.vparts + ((long long)blockIdx.y * gridDim.x + blockIdx.x) * (2 * m + 1);
    if (threadIdx.x < 2 * m) {
        const int q = threadIdx.x / m, col = threadIdx.x % m;
        double v = 0.0;
        for (int l = 0; l < rows_per_pass; l++) v += sR[q][l * m + col];
        vp[q * m + col] = v;
    } else if (threadIdx.x == 2 * m) {
        double v = 0.0;
        for (int l = 0; l < BT_THREADS; l++) v += sR[2][l];
        vp[2 * m] = v;
    }
}

__global__ void ms_bt_finish_kernel(int m, int mode, double beta, int vctas, BtLayout L, int32_t* __restrict__ n_iter,
                                    double* __restrict__ err, double* __restrict__ vaf) {
    __shared__ double s_cols[2 * BT_MAX_M + 1];
    const int p = blockIdx.x;
    const double* vp = L.vparts + (long long)p * vctas * (2 * m + 1);
    for (int e = threadIdx.x; e < 2 * m + 1; e += blockDim.x) {
        double v = 0.0;
        for (int c = 0; c < vctas; c++) v += vp[(long long)c * (2 * m + 1) + e];
        s_cols[e] = v;
    }
    __syncthreads();
    for (int j = threadIdx.x; j < m; j += blockDim.x) vaf[(long long)p * (m + 1) + 1 + j] = 1.0 - s_cols[j] / s_cols[m + j];
    if (threadIdx.x == 0) {
        double r2 = 0.0, c2 = 0.0;
        for (int j = 0; j < m; j++) r2 += s_cols[j], c2 += s_cols[m + j];
        vaf[(long long)p * (m + 1)] = 1.0 - r2 / c2;
        err[p] = bt_err(mode, s_cols[2 * m], beta);
        n_iter[p] = L.states[p].n_iter;
    }
}

// ---------------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------------
extern "C" int64_t ms_nmf_beta_workspace_bytes(int64_t n, int32_t m, int32_t n_problems, int32_t kmax) {
    if (n < 1 || m < 1 || m > BT_MAX_M || n_problems < 0 || kmax < 1 || kmax > BT_MAX_K) return 0;
    if (n_problems == 0) return 256;
    return (int64_t)bt_layout(n, m, n_problems, kmax, nullptr, nullptr) + 256;
}

#define BT_MODE_SWITCH(MODEEXPR, CALL)                                                                                \
    switch (MODEEXPR) {                                                                                               \
        case BT_IS: CALL(BT_IS); break;                                                                               \
        case BT_KL: CALL(BT_KL); break;                                                                               \
        default: CALL(BT_GEN); break;                                                                                 \
    }

extern "C" int ms_nmf_beta(const double* d_X, int64_t n, int32_t m, int64_t row_stride, int64_t col_stride,
                           const void* d_table, int32_t n_problems, int32_t kmax, double* d_W, double* d_H, double beta,
                           int32_t update_H, int32_t max_iter, double tol, int32_t regime, void* d_work,
                           int32_t* d_n_iter, double* d_err, double* d_vaf, void* stream) {
    if (!d_X || !d_table || !d_W || !d_H || !d_n_iter || !d_err || !d_vaf) return MS_E_INVALID;
    if (n < 1 || m < 1 || m > BT_MAX_M || kmax < 1 || kmax > BT_MAX_K || n_problems < 0 || max_iter < 0 ||
        !(tol >= 0.0) || !(beta == beta) || beta == 2.0 || (regime != 0 && regime != 1) || row_stride < 0 ||
        col_stride < 0 || (update_H != 0 && update_H != 1))
        return MS_E_INVALID;  // beta = 2 (Frobenius) is the job of ms_nmf_mu_* / ms_nmf_fixed_h
    if (n_problems == 0) return MS_OK;
    const int mode = beta == 1.0 ? BT_KL : beta == 0.0 ? BT_IS : BT_GEN;
    const double gamma = beta < 1.0 ? 1.0 / (2.0 - beta) : beta > 2.0 ? 1.0 / (beta - 1.0) : 1.0;
    cudaStream_t st = (cudaStream_t)stream;
    const MsNmfProblem* d_problems = (const MsNmfProblem*)d_table;
    if (regime == 0) {
        if (n > ms_nmf_beta_resident_max_rows(m, kmax)) return MS_E_INVALID;  // too long for shared memory
        const size_t smem = sizeof(double) * ((size_t)n * bt_resident_row(m, kmax) + bt_resident_fixed(m, kmax));
#define BT_LAUNCH_RESIDENT(MM)                                                                                        \
    MS_CUDA_CHECK(cudaFuncSetAttribute(ms_bt_resident_kernel<MM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    ms_bt_resident_kernel<MM><<<n_problems, BT_THREADS, smem, st>>>(d_X, (int)n, m, row_stride, col_stride, d_problems,  \
                                                                    d_W, d_H, beta, gamma, update_H, max_iter, tol,    \
                                                                    d_n_iter, d_err, d_vaf)
        BT_MODE_SWITCH(mode, BT_LAUNCH_RESIDENT)
#undef BT_LAUNCH_RESIDENT
        MS_COUNT_LAUNCH();
        MS_CUDA_CHECK(cudaGetLastError());
        return MS_OK;
    }
    if (!d_work) return MS_E_INVALID;
    BtLayout L;
    bt_layout(n, m, n_problems, kmax, (char*)d_work, &L);
    const int ctas = (int)bt_ctas(n, m, kmax, n_problems), vctas = (int)bt_vaf_ctas(n, m, n_problems);
    const int TR = bt_tile_rows(m, kmax);
    const size_t smem = bt_pass_smem(m, kmax);
#define BT_SET_SMEM(MM) MS_CUDA_CHECK(cudaFuncSetAttribute(ms_bt_pass_kernel<MM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem))
    BT_MODE_SWITCH(mode, BT_SET_SMEM)
#undef BT_SET_SMEM
    ms_bt_init_kernel<<<(n_problems + 127) / 128, 128, 0, st>>>(n_problems, max_iter, tol, L);
    MS_COUNT_LAUNCH();
    MsBtState* h_states = (MsBtState*)malloc(sizeof(MsBtState) * (size_t)n_problems);
    if (!h_states) return MS_E_INVALID;
    for (int it = 1; it <= max_iter; it++) {
#define BT_LAUNCH_PASS(MM)                                                                                            \
    ms_bt_pass_kernel<MM><<<dim3(ctas, n_problems), BT_THREADS, smem, st>>>(d_X, n, m, row_stride, col_stride,        \
                                                                            d_problems, d_W, d_H, beta, gamma,        \
                                                                            update_H, TR, L, kmax)
        BT_MODE_SWITCH(mode, BT_LAUNCH_PASS)
#undef BT_LAUNCH_PASS
        MS_COUNT_LAUNCH();
        ms_bt_update_kernel<<<n_problems, BT_THREADS, 0, st>>>(d_problems, d_H, m, mode, beta, gamma, update_H, it,
                                                               max_iter, tol, ctas, L, kmax);
        MS_COUNT_LAUNCH();
        if (tol > 0.0 && it % 64 == 0 && it < max_iter) {
            // stop early once every problem is done (pageable copy: waits for the stream)
            cudaError_t e = cudaMemcpyAsync(h_states, L.states, sizeof(MsBtState) * (size_t)n_problems,
                                            cudaMemcpyDeviceToHost, st);
            if (e == cudaSuccess) e = cudaStreamSynchronize(st);
            if (e != cudaSuccess) {
                free(h_states);
                MS_CUDA_CHECK(e);
            }
            int all_done = 1;
            for (int p = 0; p < n_problems; p++) all_done &= h_states[p].done != 0;
            if (all_done) break;
        }
    }
    free(h_states);
    ms_bt_restore_kernel<<<dim3(ctas, n_problems), BT_THREADS, 0, st>>>(n, d_problems, d_W, L, kmax);
    MS_COUNT_LAUNCH();
#define BT_LAUNCH_FINAL(MM)                                                                                           \
    ms_bt_final_kernel<MM><<<dim3(vctas, n_problems), BT_THREADS, 0, st>>>(d_X, n, m, row_stride, col_stride,         \
                                                                           d_problems, d_W, d_H, beta, L)
    BT_MODE_SWITCH(mode, BT_LAUNCH_FINAL)
#undef BT_LAUNCH_FINAL
    MS_COUNT_LAUNCH();
    ms_bt_finish_kernel<<<n_problems, 64, 0, st>>>(m, mode, beta, vctas, L, d_n_iter, d_err, d_vaf);
    MS_COUNT_LAUNCH();
    MS_CUDA_CHECK(cudaGetLastError());
    return MS_OK;
}
