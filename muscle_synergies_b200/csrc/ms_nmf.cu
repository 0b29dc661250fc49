// Batched NMF by multiplicative updates (Frobenius loss) - EXTENSION stage.
//
// The reference only wraps scikit-learn here: find_synergies -> NMF(n_components=k, **kwargs)
// .fit_transform(X) (src/muscle_synergies/analysis.py:848-882) and vaf (:597-667).  This file
// implements, for solver="mu", beta_loss="frobenius", the update sklearn executes
// (sklearn/decomposition/_nmf.py, _fit_multiplicative_update; SURVEY.md Appendix E):
//
//     W <- W * (X H^T) / (W (H H^T))      denominators == 0 replaced by EPS (float32 eps)
//     H <- H * (W^T X) / ((W^T W) H)      with the UPDATED W
//     every `check_every` iterations (tol > 0): e = ||X - W H||_F ; stop if (prev - e) / e0 < tol
//
// in fp32 for a whole batch of problems (rank sweep x random restarts) per launch.  It is
// checked against sklearn within a stated tolerance (tests/test_nmf_gpu.py); it is not a
// bit-parity claim.
//
//   ms_nmf_resident_kernel   one CTA per problem, X / W / H resident in shared memory for the
//                            whole run (the 200 x 16 envelopes of the reference flow are 12.8 KB):
//                            no HBM traffic between iterations, bound by SM issue + shared memory
//   ms_nmf_stream_*          long signals: X and W stream from HBM once per iteration, W^T X and
//                            W^T W reduced per CTA and accumulated with atomics (HBM-bound)
#include "ms_nmf_common.cuh"

#define NMF_EPS 1.1920929e-07f
// The quotient of an update step: one reciprocal approximation and a multiply (2 ulp) instead of the ~10 instructions of
// an IEEE division - the iteration is self-correcting and the stated tolerance against scikit-learn (1e-4 in VAF) is five
// orders of magnitude above it.  -DNMF_IEEE_DIV restores the exact quotient.  Same-box A/B (tools/time_nmf.py), together
// with skipping the arithmetic on padding components: 48.9 -> 55.1 M it/s (160 problems), 80.5 -> 94.2 M it/s (1280).
#ifdef NMF_IEEE_DIV
#define NMF_DIV(a, b) ((a) / (b))
#else
#define NMF_DIV(a, b) __fdividef((a), (b))
#endif
#define NMF_THREADS 256
#ifndef NMF_MIN_CTAS
#define NMF_MIN_CTAS 3
#endif

__device__ __forceinline__ float ms_block_sum(float v, float* s_red) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) s_red[warp] = v;
    __syncthreads();
    float t = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) t += s_red[w];
    return t;
}

// ---------------------------------------------------------------------------------------------------
// resident regime
// ---------------------------------------------------------------------------------------------------
struct MsNmfArgs {
    const float* X;
    int n, m;
    float* Wp;
    float* Hp;
    int max_iter;
    float tol;
    int check_every;
    int32_t* n_iter_out;
    float* err_out;
    float* vaf_out;  // [m + 1] of this problem
};

// Shared-memory layout of one problem (floats; every row 16-byte aligned so that rows are read as float4):
//   sX   [n][XS]   X, columns padded with zeros to MP = roundup(m, 4); XS = MP or MP + 4 so that XS / 4 is odd
//                  (a quarter warp reading one float4 per row then touches 8 different bank groups)
//   sW   [n][WS]   W, columns padded with zeros to KP = roundup(K, 4); WS likewise
//   sHt  [MP][KP]  H transposed (rows past m are zero): the K weights of muscle j are one or more float4 (W step, residual)
//   sH   [K][MP]   H (H step, H H^T)
//   sHHt [K][KP], sWtW [KP][KP], sWtX [KP][MP], sPart [slices][tiles * 16], s_red [32]
__host__ __device__ inline int ms_nmf_pad4(int v) { return (v + 3) & ~3; }
__host__ __device__ inline int ms_nmf_stride(int padded) { return ((padded >> 2) & 1) ? padded : padded + 4; }

// element e of the 4 x 4 tile list (W^T W tiles, then W^T X tiles) -> its place in sWtW / sWtX
template <int K>
__device__ __forceinline__ float* ms_nmf_tile_dst(int e, int MQ, int MP, float* sWtW, float* sWtX) {
    constexpr int KP = (K + 3) & ~3, KQ = KP / 4;
    const int tile = e >> 4, r = (e >> 2) & 3, c = e & 3;
    if (tile < KQ * KQ) return sWtW + (4 * (tile / KQ) + r) * KP + 4 * (tile % KQ) + c;
    const int q = tile - KQ * KQ;
    return sWtX + (4 * (q / MQ) + r) * MP + 4 * (q % MQ) + c;
}

template <int K>
__device__ __forceinline__ void ms_nmf_resident_body(const MsNmfArgs& A, float* sm) {
    constexpr int KP = (K + 3) & ~3, KQ = KP / 4;
    constexpr int WS = ((KP >> 2) & 1) ? KP : KP + 4;
    const int n = A.n, m = A.m;
    const int MP = ms_nmf_pad4(m), MQ = MP / 4, XS = ms_nmf_stride(MP);
    const int n_tiles = KQ * KQ + KQ * MQ;  // 4 x 4 output tiles of W^T W and W^T X
    int slices = NMF_THREADS / n_tiles;     // row slices that work on the tiles side by side
    if (slices < 1) slices = 1;
    if (slices > n) slices = n;
    float* sX = sm;
    float* sW = sX + n * XS;
    float* sHt = sW + n * WS;
    float* sH = sHt + MP * KP;
    float* sHHt = sH + K * MP;
    float* sWtW = sHHt + K * KP;
    float* sWtX = sWtW + KP * KP;
    float* sPart = sWtX + KP * MP;
    float* s_red = sPart + NMF_THREADS * 16;
    const int tid = threadIdx.x;

    for (int i = tid; i < n * XS; i += NMF_THREADS) {
        const int r = i / XS, c = i - r * XS;
        sX[i] = c < m ? A.X[r * m + c] : 0.f;
    }
    for (int i = tid; i < n * WS; i += NMF_THREADS) {
        const int r = i / WS, c = i - r * WS;
        sW[i] = c < K ? A.Wp[r * K + c] : 0.f;
    }
    for (int i = tid; i < K * MP; i += NMF_THREADS) {
        const int a = i / MP, j = i - a * MP;
        sH[i] = j < m ? A.Hp[a * m + j] : 0.f;
    }
    for (int i = tid; i < MP * KP; i += NMF_THREADS) {
        const int j = i / KP, a = i - j * KP;
        sHt[i] = (a < K && j < m) ? A.Hp[a * m + j] : 0.f;
    }
    // the padding of H H^T must read as zero: the W step runs over whole float4 groups of components
    for (int i = tid; i < K * KP; i += NMF_THREADS) sHHt[i] = 0.f;
    __syncthreads();

    // sum over the rows this thread owns of |x_i - w_i H|^2
    auto residual_sq = [&]() {
        double acc = 0.0;
        for (int i = tid; i < n; i += NMF_THREADS) {
            float w[KP];
#pragma unroll
            for (int q = 0; q < KQ; q++) {
                const float4 v = *reinterpret_cast<const float4*>(sW + i * WS + 4 * q);
                w[4 * q] = v.x, w[4 * q + 1] = v.y, w[4 * q + 2] = v.z, w[4 * q + 3] = v.w;
            }
            for (int j = 0; j < m; j++) {
                float r = sX[i * XS + j];
#pragma unroll
                for (int q = 0; q < KQ; q++) {
                    const float4 h = *reinterpret_cast<const float4*>(sHt + j * KP + 4 * q);
                    r = fmaf(-w[4 * q], h.x, r);
                    r = fmaf(-w[4 * q + 1], h.y, r);
                    r = fmaf(-w[4 * q + 2], h.z, r);
                    r = fmaf(-w[4 * q + 3], h.w, r);
                }
                acc += (double)r * (double)r;
            }
        }
        // summed in double: the stop test compares residuals that differ in the sixth digit (tol = 1e-6 is the
        // reference's default, analysis.py:718-719); float sums over n*m terms carry roundoff of that order
        return ms_block_sum_d(acc, reinterpret_cast<double*>(s_red));
    };
    auto compute_hht = [&]() {
        for (int e = tid; e < K * K; e += NMF_THREADS) {
            const int a = e / K, b = e % K;
            // rows of H as float4 (the zero padding adds nothing), two accumulators
            float acc0 = 0.f, acc1 = 0.f;
            for (int jq = 0; jq < MQ; jq++) {
                const float4 u = *reinterpret_cast<const float4*>(sH + a * MP + 4 * jq);
                const float4 v = *reinterpret_cast<const float4*>(sH + b * MP + 4 * jq);
                acc0 = fmaf(u.x, v.x, acc0);
                acc1 = fmaf(u.y, v.y, acc1);
                acc0 = fmaf(u.z, v.z, acc0);
                acc1 = fmaf(u.w, v.w, acc1);
            }
            const float acc = acc0 + acc1;
            sHHt[a * KP + b] = acc;
        }
    };

    double err0 = 0.0, prev = 0.0;
    if (A.tol > 0.f) {
        err0 = sqrt(residual_sq());
        prev = err0;
    }
    compute_hht();
    __syncthreads();

    // index arithmetic that does not change from one iteration to the next
    const bool t2_active = tid < n_tiles * slices;
    const float* t2_left = sW;   // 4 columns of W
    const float* t2_right = sW;  // 4 columns of W (tile of W^T W) or of X (tile of W^T X)
    int t2_rstride = WS, t2_i0 = 0, t2_i1 = 0;
    float* t2_part = sPart;
    if (t2_active) {
        const int tile = tid % n_tiles, sl = tid / n_tiles;
        const int rows_per = (n + slices - 1) / slices;
        t2_i0 = sl * rows_per;
        t2_i1 = min(n, t2_i0 + rows_per);
        if (tile < KQ * KQ) {
            t2_left = sW + 4 * (tile / KQ);
            t2_right = sW + 4 * (tile % KQ);
        } else {
            const int q = tile - KQ * KQ;
            t2_left = sW + 4 * (q / MQ);
            t2_right = sX + 4 * (q % MQ);
            t2_rstride = XS;
        }
        t2_part = sPart + (sl * n_tiles + tile) * 16;
    }
    // where this thread's first reduced tile element goes (usually its only one)
    float* t2_dst0 = ms_nmf_tile_dst<K>(min(tid, n_tiles * 16 - 1), MQ, MP, sWtW, sWtX);

    int it = 0;
    for (it = 1; it <= A.max_iter; it++) {
        // ---- W <- W * (X H^T) / (W (H H^T)): one row per thread, H^T and H H^T read as broadcast float4
        for (int i = tid; i < n; i += NMF_THREADS) {
            float w[KP], num[KP], den[KP];
#pragma unroll
            for (int q = 0; q < KQ; q++) {
                const float4 v = *reinterpret_cast<const float4*>(sW + i * WS + 4 * q);
                w[4 * q] = v.x, w[4 * q + 1] = v.y, w[4 * q + 2] = v.z, w[4 * q + 3] = v.w;
            }
#pragma unroll
            for (int c = 0; c < KP; c++) num[c] = den[c] = 0.f;
            for (int jq = 0; jq < MQ; jq++) {
                const float4 xv = *reinterpret_cast<const float4*>(sX + i * XS + 4 * jq);
                const float x4[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
                for (int jj = 0; jj < 4; jj++) {
                    const float* ht = sHt + (4 * jq + jj) * KP;  // rows past m exist and are zero, like x there
#pragma unroll
                    for (int q = 0; q < KQ; q++) {
                        // components past K are padding: no arithmetic on them (the conditions fold at compile time)
                        const float4 h = *reinterpret_cast<const float4*>(ht + 4 * q);
                        num[4 * q] = fmaf(x4[jj], h.x, num[4 * q]);
                        if (4 * q + 1 < K) num[4 * q + 1] = fmaf(x4[jj], h.y, num[4 * q + 1]);
                        if (4 * q + 2 < K) num[4 * q + 2] = fmaf(x4[jj], h.z, num[4 * q + 2]);
                        if (4 * q + 3 < K) num[4 * q + 3] = fmaf(x4[jj], h.w, num[4 * q + 3]);
                    }
                }
            }
#pragma unroll
            for (int b = 0; b < K; b++) {
#pragma unroll
                for (int q = 0; q < KQ; q++) {
                    const float4 g = *reinterpret_cast<const float4*>(sHHt + b * KP + 4 * q);
                    den[4 * q] = fmaf(w[b], g.x, den[4 * q]);
                    if (4 * q + 1 < K) den[4 * q + 1] = fmaf(w[b], g.y, den[4 * q + 1]);
                    if (4 * q + 2 < K) den[4 * q + 2] = fmaf(w[b], g.z, den[4 * q + 2]);
                    if (4 * q + 3 < K) den[4 * q + 3] = fmaf(w[b], g.w, den[4 * q + 3]);
                }
            }
#pragma unroll
            for (int c = 0; c < K; c++) {
                const float d = den[c] == 0.f ? NMF_EPS : den[c];
                w[c] = w[c] * NMF_DIV(num[c], d);  // padding components stay 0
            }
#pragma unroll
            for (int q = 0; q < KQ; q++)
                *reinterpret_cast<float4*>(sW + i * WS + 4 * q) = make_float4(w[4 * q], w[4 * q + 1], w[4 * q + 2], w[4 * q + 3]);
        }
        __syncthreads();
        // ---- W^T W and W^T X: 4 x 4 register tiles, the rows split into slices that run side by side
        if (t2_active) {
            float acc[4][4];
#pragma unroll
            for (int r = 0; r < 4; r++)
#pragma unroll
                for (int c = 0; c < 4; c++) acc[r][c] = 0.f;
#pragma unroll 2
            for (int i = t2_i0; i < t2_i1; i++) {
                const float4 a = *reinterpret_cast<const float4*>(t2_left + i * WS);
                const float4 b = *reinterpret_cast<const float4*>(t2_right + i * t2_rstride);
                const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
                for (int r = 0; r < 4; r++)
#pragma unroll
                    for (int c = 0; c < 4; c++) acc[r][c] = fmaf(av[r], bv[c], acc[r][c]);
            }
#pragma unroll
            for (int r = 0; r < 4; r++) *reinterpret_cast<float4*>(t2_part + 4 * r) = make_float4(acc[r][0], acc[r][1], acc[r][2], acc[r][3]);
        }
        __syncthreads();
        for (int e = tid; e < n_tiles * 16; e += NMF_THREADS) {
            // four independent partial sums: the loads of a dependent chain would each wait for the last add
            float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
            const int stride = n_tiles * 16;
            int sl = 0;
            for (; sl + 4 <= slices; sl += 4) {
                a0 += sPart[sl * stride + e];
                a1 += sPart[(sl + 1) * stride + e];
                a2 += sPart[(sl + 2) * stride + e];
                a3 += sPart[(sl + 3) * stride + e];
            }
            for (; sl < slices; sl++) a0 += sPart[sl * stride + e];
            *(e == tid ? t2_dst0 : ms_nmf_tile_dst<K>(e, MQ, MP, sWtW, sWtX)) = (a0 + a1) + (a2 + a3);
        }
        __syncthreads();
        // ---- H <- H * (W^T X) / ((W^T W) H)
        {
            float newh[(MS_NMF_MAX_K * MS_NMF_MAX_M + NMF_THREADS - 1) / NMF_THREADS];
            int q = 0;
            for (int e = tid; e < K * m; e += NMF_THREADS, q++) {
                const int a = e / m, j = e - a * m;
                float den = 0.f;
#pragma unroll
                for (int b = 0; b < K; b++) den = fmaf(sWtW[a * KP + b], sH[b * MP + j], den);
                if (den == 0.f) den = NMF_EPS;
                newh[q] = sH[a * MP + j] * NMF_DIV(sWtX[a * MP + j], den);
            }
            __syncthreads();
            q = 0;
            for (int e = tid; e < K * m; e += NMF_THREADS, q++) {
                const int a = e / m, j = e - a * m;
                sH[a * MP + j] = newh[q];
                sHt[j * KP + a] = newh[q];
            }
        }
        __syncthreads();
        compute_hht();
        __syncthreads();
        if (A.tol > 0.f && it % A.check_every == 0) {
            const double err = sqrt(residual_sq());
            if (err0 == 0.0 || (prev - err) / err0 < (double)A.tol) break;  // an exactly factorised X has converged
            prev = err;
        }
    }
    if (it > A.max_iter) it = A.max_iter;

    // ---- results: factors, ||X - W H||_F, variance accounted for (analysis.py:642-667)
    for (int i = tid; i < n * K; i += NMF_THREADS) A.Wp[i] = sW[(i / K) * WS + (i % K)];
    for (int i = tid; i < K * m; i += NMF_THREADS) A.Hp[i] = sH[(i / m) * MP + (i % m)];
    const float res = (float)residual_sq();
    float xx = 0.f;
    for (int i = tid; i < n * m; i += NMF_THREADS) {
        const float v = sX[(i / m) * XS + (i % m)];
        xx = fmaf(v, v, xx);
    }
    xx = ms_block_sum(xx, s_red);
    if (tid == 0) {
        *A.n_iter_out = it;
        *A.err_out = sqrtf(res);
        A.vaf_out[0] = 1.f - res / xx;
    }
    // per-muscle VAF: one column per thread
    for (int j = tid; j < m; j += NMF_THREADS) {
        float rs = 0.f, cs = 0.f;
        for (int i = 0; i < n; i++) {
            float r = sX[i * XS + j];
            cs = fmaf(r, r, cs);
#pragma unroll
            for (int c = 0; c < K; c++) r = fmaf(-sW[i * WS + c], sH[c * MP + j], r);
            rs = fmaf(r, r, rs);
        }
        A.vaf_out[1 + j] = 1.f - rs / cs;
    }
}

__global__ void __launch_bounds__(NMF_THREADS, NMF_MIN_CTAS)
    ms_nmf_resident_kernel(const float* __restrict__ X, int n, int m, const MsNmfProblem* __restrict__ problems,
                           float* __restrict__ Wg, float* __restrict__ Hg, int max_iter, float tol, int check_every,
                           int32_t* __restrict__ n_iter_out, float* __restrict__ err_out, float* __restrict__ vaf_out) {
    extern __shared__ float sm[];
    const MsNmfProblem pb = problems[blockIdx.x];
    MsNmfArgs A;
    A.X = X + pb.x_off;
    A.n = n;
    A.m = m;
    A.Wp = Wg + pb.w_off;
    A.Hp = Hg + pb.h_off;
    A.max_iter = max_iter;
    A.tol = tol;
    A.check_every = check_every;
    A.n_iter_out = n_iter_out + blockIdx.x;
    A.err_out = err_out + blockIdx.x;
    A.vaf_out = vaf_out + (long long)blockIdx.x * (m + 1);
#define NMF_RESIDENT(KK) ms_nmf_resident_body<KK>(A, sm)
    MS_NMF_K_SWITCH(pb.k, NMF_RESIDENT)
#undef NMF_RESIDENT
}

static size_t ms_nmf_resident_fixed_floats(int m, int kmax) {
    const int KP = ms_nmf_pad4(kmax), MP = ms_nmf_pad4(m);
    return (size_t)MP * KP + (size_t)kmax * MP + (size_t)kmax * KP + (size_t)KP * KP + (size_t)KP * MP +
           (size_t)NMF_THREADS * 16 + 32;
}
static size_t ms_nmf_resident_row_floats(int m, int kmax) {
    return (size_t)ms_nmf_stride(ms_nmf_pad4(m)) + (size_t)ms_nmf_stride(ms_nmf_pad4(kmax));
}
static size_t ms_nmf_resident_smem(int n, int m, int kmax) {
    return sizeof(float) * ((size_t)n * ms_nmf_resident_row_floats(m, kmax) + ms_nmf_resident_fixed_floats(m, kmax));
}

// Largest n the resident kernel takes for (m, kmax); 0 if the shape is unsupported.
extern "C" int32_t ms_nmf_resident_max_rows(int32_t m, int32_t kmax) {
    return ms_nmf_max_rows(m, kmax, sizeof(float), ms_nmf_resident_fixed_floats, ms_nmf_resident_row_floats);
}

// The problem table of a batch (32 bytes per problem: rank, offsets of its W, H and X), written to HOST memory the
// caller owns; returns the largest rank, or a negative MS_E_* code.  A caller that runs the same sweep again and again
// (one launch per trial) copies the table to the device once and then uses ms_nmf_mu_batched_planned, which neither
// copies nor waits.
extern "C" int32_t ms_nmf_plan(int32_t n, int32_t m, const int32_t* h_ranks, const int32_t* h_x_index, int32_t n_problems,
                               void* h_table) {
    if (!h_ranks || !h_table || n < 1 || m < 1 || m > MS_NMF_MAX_M || n_problems < 0) return MS_E_INVALID;
    return ms_nmf_fill_table(n, m, h_ranks, h_x_index, n_problems, (MsNmfProblem*)h_table);
}

// The table of ms_nmf_plan, copied to d_table (and waited for); returns the largest rank or a negative MS_E_* code.
static int ms_nmf_upload_table(long long n, int m, const int32_t* h_ranks, const int32_t* h_x_index, int n_problems,
                               void* d_table, cudaStream_t st) {
    MsNmfProblem* h = (MsNmfProblem*)malloc(sizeof(MsNmfProblem) * n_problems);
    if (!h) return MS_E_INVALID;
    const int kmax = ms_nmf_fill_table(n, m, h_ranks, h_x_index, n_problems, h);
    cudaError_t e = cudaSuccess;
    if (kmax > 0) {
        e = cudaMemcpyAsync(d_table, h, sizeof(MsNmfProblem) * n_problems, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);  // h is pageable: do not free it under the copy
    }
    free(h);
    MS_CUDA_CHECK(e);
    return kmax;
}

// ms_nmf_mu_batched with the table of ms_nmf_plan already in device memory: one launch, nothing else.
extern "C" int ms_nmf_mu_batched_planned(const float* d_X, int32_t n, int32_t m, const void* d_table, int32_t n_problems,
                                         int32_t kmax, float* d_W, float* d_H, int32_t max_iter, float tol,
                                         int32_t check_every, int32_t* d_n_iter, float* d_err, float* d_vaf, void* stream) {
    if (!d_X || !d_table || !d_W || !d_H || !d_n_iter || !d_err || !d_vaf) return MS_E_INVALID;
    if (n < 1 || m < 1 || m > MS_NMF_MAX_M || kmax < 1 || kmax > MS_NMF_MAX_K || n_problems < 0 || max_iter < 0 || check_every < 1)
        return MS_E_INVALID;
    if (n_problems == 0) return MS_OK;
    if (n > ms_nmf_resident_max_rows(m, kmax)) return MS_E_INVALID;  // too long for the resident kernel: use ms_nmf_mu_stream
    cudaStream_t st = (cudaStream_t)stream;
    const size_t smem = ms_nmf_resident_smem(n, m, kmax);
    MS_CUDA_CHECK(cudaFuncSetAttribute(ms_nmf_resident_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ms_nmf_resident_kernel<<<n_problems, NMF_THREADS, smem, st>>>(d_X, n, m, (const MsNmfProblem*)d_table, d_W, d_H, max_iter,
                                                                  tol, check_every, d_n_iter, d_err, d_vaf);
    MS_COUNT_LAUNCH();
    MS_CUDA_CHECK(cudaGetLastError());
    return MS_OK;
}

// h_ranks[P]: rank of each problem; h_x_index[P] (may be NULL = all 0): which [n][m] matrix of d_X
// problem p factorises.  d_W / d_H hold the initial factors packed problem after problem (W_p is
// [n][k_p] row-major, H_p is [k_p][m]) and receive the results in place.
// d_work: P * 32 bytes.  d_vaf: [P][m + 1] (overall, then per column).
extern "C" int ms_nmf_mu_batched(const float* d_X, int32_t n, int32_t m, const int32_t* h_ranks,
                                 const int32_t* h_x_index, int32_t n_problems,
                                 float* d_W, float* d_H, int32_t max_iter, float tol, int32_t check_every, void* d_work,
                                 int32_t* d_n_iter, float* d_err, float* d_vaf, void* stream) {
    if (!d_X || !h_ranks || !d_W || !d_H || !d_work || !d_n_iter || !d_err || !d_vaf) return MS_E_INVALID;
    if (n < 1 || m < 1 || m > MS_NMF_MAX_M || n_problems < 0 || max_iter < 0 || check_every < 1) return MS_E_INVALID;
    if (n_problems == 0) return MS_OK;
    const int kmax = ms_nmf_upload_table(n, m, h_ranks, h_x_index, n_problems, d_work, (cudaStream_t)stream);
    if (kmax < 0) return kmax;
    return ms_nmf_mu_batched_planned(d_X, n, m, d_work, n_problems, kmax, d_W, d_H, max_iter, tol, check_every, d_n_iter,
                                     d_err, d_vaf, stream);
}

// ---------------------------------------------------------------------------------------------------
// streaming regime: X and W too long for shared memory
// ---------------------------------------------------------------------------------------------------
// Per iteration and problem, X [n][m] and W [n][k] stream through HBM exactly once:
//   ms_nmf_stream_w_kernel   each CTA loops over 256-row tiles: tile of X and W -> shared memory
//                            (coalesced), W rows updated with the problem's H and H H^T, tile written
//                            back, and the tile's contribution to W^T X and W^T W accumulated in
//                            registers; one atomicAdd per CTA and output at the end
//   ms_nmf_stream_h_kernel   one small CTA per problem: H update, H H^T for the next iteration, the
//                            objective from ||X||^2 - 2 <H, W^T X> + <W^T W, H H^T> (no extra pass over X)
// Algorithmic bytes per iteration and problem: 4 n m (X) + 8 n k (W read + write).
#define NMFS_ROWS 256

struct MsNmfStreamState {  // per problem, device memory
    float HHt[MS_NMF_MAX_K * MS_NMF_MAX_K];
    float acc[MS_NMF_MAX_K * MS_NMF_MAX_K + MS_NMF_MAX_K * MS_NMF_MAX_M];  // W^T W then W^T X
    float err0, prev, err;
    int n_iter, done;
};

// One pass over X and W for one problem: per 256-row tile, stage X and W (float4 rows, same padded layout
// as the resident kernel), update the W rows (one row per thread, H^T and H H^T as broadcast float4), write them
// back, and accumulate W^T W / W^T X in a 4 x 4 register tile that lives across all the tiles a CTA visits -
// shared memory is read as float4 only, and the reduction happens once, at the end, with global atomics.
// The tiles are double-buffered: the 16-byte asynchronous copies (cp.async) of the next tile are in flight while
// this one is computed, so the pass runs at memory speed instead of waiting out a round trip per tile.
__device__ __forceinline__ void ms_cp_async16(void* smem_dst, const void* gmem_src) {
    const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(gmem_src) : "memory");
}

template <int K>
__device__ __forceinline__ void ms_nmf_stream_w_body(const float* __restrict__ X, long long n, int m, float* __restrict__ Wp,
                                                     const float* __restrict__ Hp, MsNmfStreamState* __restrict__ stt,
                                                     float* sm) {
    constexpr int KP = (K + 3) & ~3, KQ = KP / 4;
    constexpr int WS = ((KP >> 2) & 1) ? KP : KP + 4;
    const int MP = ms_nmf_pad4(m), MQ = MP / 4, XS = ms_nmf_stride(MP);
    float* sXb = sm;                          // [2][NMFS_ROWS][XS]
    float* sWb = sXb + 2 * NMFS_ROWS * XS;    // [2][NMFS_ROWS][WS]
    float* sHt = sWb + 2 * NMFS_ROWS * WS;    // [MP][KP]
    float* sHHt = sHt + MP * KP;              // [K][KP]
    const int tid = threadIdx.x;
    for (int i = tid; i < 2 * NMFS_ROWS * XS; i += NMFS_ROWS) sXb[i] = 0.f;  // the padding columns stay zero
    for (int i = tid; i < 2 * NMFS_ROWS * WS; i += NMFS_ROWS) sWb[i] = 0.f;
    for (int i = tid; i < MP * KP; i += NMFS_ROWS) {
        const int j = i / KP, c = i - j * KP;
        sHt[i] = (c < K && j < m) ? Hp[c * m + j] : 0.f;
    }
    for (int i = tid; i < K * KP; i += NMFS_ROWS) {
        const int bq = i / KP, c = i - bq * KP;
        sHHt[i] = c < K ? stt->HHt[bq * K + c] : 0.f;
    }
    // this thread's 4 x 4 tile of W^T W or W^T X and its slice of the rows of every tile
    // (at most 4 * 4 + 4 * 16 = 80 tiles for k <= 16, m <= 64: one per thread is enough)
    const int n_tiles4 = KQ * KQ + KQ * MQ;
    const int slices = NMFS_ROWS / n_tiles4;
    const int rows_per = (NMFS_ROWS + slices - 1) / slices;
    const bool t2_active = tid < n_tiles4 * slices;
    const int t4 = tid % n_tiles4, t2_i0 = (tid / n_tiles4) * rows_per;
    int t2_left = 0, t2_right = 0, t2_rstride = WS;  // offsets inside the W / X buffers
    bool t2_x = false;
    if (t4 < KQ * KQ) {
        t2_left = 4 * (t4 / KQ);
        t2_right = 4 * (t4 % KQ);
    } else {
        const int q = t4 - KQ * KQ;
        t2_left = 4 * (q / MQ);
        t2_right = 4 * (q % MQ);
        t2_rstride = XS;
        t2_x = true;
    }
    float acc[4][4];
#pragma unroll
    for (int r = 0; r < 4; r++)
#pragma unroll
        for (int c = 0; c < 4; c++) acc[r][c] = 0.f;
    // float4 global accesses need 16-byte aligned rows: whole float4 groups per row and an aligned base (a
    // problem's W starts wherever the previous problems' factors end)
    const bool vec_x = (m & 3) == 0 && (reinterpret_cast<uintptr_t>(X) & 15) == 0;
    const bool vec_w = (K & 3) == 0 && (reinterpret_cast<uintptr_t>(Wp) & 15) == 0;
    const long long n_tiles = (n + NMFS_ROWS - 1) / NMFS_ROWS;

    auto prefetch = [&](long long tile, int buf) {  // the aligned parts of a tile, asynchronously
        if (tile < n_tiles) {
            const long long r0 = tile * NMFS_ROWS;
            const int rows = (int)min((long long)NMFS_ROWS, n - r0);
            if (vec_x) {
                const float* src = X + r0 * m;
                float* dst = sXb + buf * NMFS_ROWS * XS;
                for (int i = tid; i < rows * MQ; i += NMFS_ROWS) {
                    const int r = i / MQ, q = i - r * MQ;
                    ms_cp_async16(dst + r * XS + 4 * q, src + 4 * i);
                }
            }
            if (vec_w) {
                const float* src = Wp + r0 * K;
                float* dst = sWb + buf * NMFS_ROWS * WS;
                for (int i = tid; i < rows * KQ; i += NMFS_ROWS) {
                    const int r = i / KQ, q = i - r * KQ;
                    ms_cp_async16(dst + r * WS + 4 * q, src + 4 * i);
                }
            }
        }
        asm volatile("cp.async.commit_group;\n" ::: "memory");
    };

    __syncthreads();  // the zero fill above must not race with the first copies
    int buf = 0;
    prefetch(blockIdx.x, 0);
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, buf ^= 1) {
        const long long r0 = tile * NMFS_ROWS;
        const int rows = (int)min((long long)NMFS_ROWS, n - r0);
        float* sX = sXb + buf * NMFS_ROWS * XS;
        float* sW = sWb + buf * NMFS_ROWS * WS;
        prefetch(tile + gridDim.x, buf ^ 1);  // nobody reads that buffer any more: see the barrier at the loop's end
        if (!vec_x)
            for (int i = tid; i < rows * m; i += NMFS_ROWS) sX[(i / m) * XS + (i % m)] = X[r0 * m + i];
        if (!vec_w)
            for (int i = tid; i < rows * K; i += NMFS_ROWS) sW[(i / K) * WS + (i % K)] = Wp[r0 * K + i];
        asm volatile("cp.async.wait_group 1;\n" ::: "memory");  // this tile's copies (the next tile's may still fly)
        __syncthreads();
        if (tid < rows) {
            const int i = tid;
            float w[KP], num[KP], den[KP];
#pragma unroll
            for (int q = 0; q < KQ; q++) {
                const float4 v = *reinterpret_cast<const float4*>(sW + i * WS + 4 * q);
                w[4 * q] = v.x, w[4 * q + 1] = v.y, w[4 * q + 2] = v.z, w[4 * q + 3] = v.w;
            }
#pragma unroll
            for (int c = 0; c < KP; c++) num[c] = den[c] = 0.f;
            for (int jq = 0; jq < MQ; jq++) {
                const float4 xv = *reinterpret_cast<const float4*>(sX + i * XS + 4 * jq);
                const float x4[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
                for (int jj = 0; jj < 4; jj++) {
                    const float* ht = sHt + (4 * jq + jj) * KP;
#pragma unroll
                    for (int q = 0; q < KQ; q++) {
                        // components past K are padding: no arithmetic on them (the conditions fold at compile time)
                        const float4 h = *reinterpret_cast<const float4*>(ht + 4 * q);
                        num[4 * q] = fmaf(x4[jj], h.x, num[4 * q]);
                        if (4 * q + 1 < K) num[4 * q + 1] = fmaf(x4[jj], h.y, num[4 * q + 1]);
                        if (4 * q + 2 < K) num[4 * q + 2] = fmaf(x4[jj], h.z, num[4 * q + 2]);
                        if (4 * q + 3 < K) num[4 * q + 3] = fmaf(x4[jj], h.w, num[4 * q + 3]);
                    }
                }
            }
#pragma unroll
            for (int bq = 0; bq < K; bq++) {
#pragma unroll
                for (int q = 0; q < KQ; q++) {
                    const float4 g = *reinterpret_cast<const float4*>(sHHt + bq * KP + 4 * q);
                    den[4 * q] = fmaf(w[bq], g.x, den[4 * q]);
                    den[4 * q + 1] = fmaf(w[bq], g.y, den[4 * q + 1]);
                    den[4 * q + 2] = fmaf(w[bq], g.z, den[4 * q + 2]);
                    den[4 * q + 3] = fmaf(w[bq], g.w, den[4 * q + 3]);
                }
            }
#pragma unroll
            for (int c = 0; c < KP; c++) {
                const float d = den[c] == 0.f ? NMF_EPS : den[c];
                w[c] = w[c] * (num[c] / d);  // padding components: 0 * (0 / eps) = 0
            }
#pragma unroll
            for (int q = 0; q < KQ; q++)
                *reinterpret_cast<float4*>(sW + i * WS + 4 * q) = make_float4(w[4 * q], w[4 * q + 1], w[4 * q + 2], w[4 * q + 3]);
        }
        __syncthreads();
        if (vec_w) {
            float4* dst = reinterpret_cast<float4*>(Wp + r0 * K);
            for (int i = tid; i < rows * KQ; i += NMFS_ROWS) {
                const int r = i / KQ, q = i - r * KQ;
                dst[i] = *reinterpret_cast<const float4*>(sW + r * WS + 4 * q);
            }
        } else {
            for (int i = tid; i < rows * K; i += NMFS_ROWS) Wp[r0 * K + i] = sW[(i / K) * WS + (i % K)];
        }
        if (t2_active) {
            const float* left = sW + t2_left;
            const float* right = (t2_x ? sX : sW) + t2_right;
            const int i1 = min(rows, t2_i0 + rows_per);
#pragma unroll 2
            for (int i = t2_i0; i < i1; i++) {
                const float4 av = *reinterpret_cast<const float4*>(left + i * WS);
                const float4 bv = *reinterpret_cast<const float4*>(right + i * t2_rstride);
                const float a4[4] = {av.x, av.y, av.z, av.w}, b4[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
                for (int r = 0; r < 4; r++)
#pragma unroll
                    for (int c = 0; c < 4; c++) acc[r][c] = fmaf(a4[r], b4[c], acc[r][c]);
            }
        }
        __syncthreads();  // everyone is done with this buffer before the next iteration's copies land in it
    }
    asm volatile("cp.async.wait_group 0;\n" ::: "memory");
    // one reduction per CTA: tile element (r, c) -> W^T W [K][K], then W^T X [K][m] behind it
    if (t2_active) {
#pragma unroll
        for (int r = 0; r < 4; r++)
#pragma unroll
            for (int c = 0; c < 4; c++) {
                const int a = t2_left + r, bcol = t2_right + c;
                const int width = t2_x ? m : K, base = t2_x ? K * K : 0;
                if (a < K && bcol < width) atomicAdd(&stt->acc[base + a * width + bcol], acc[r][c]);
            }
    }
}

__global__ void __launch_bounds__(NMFS_ROWS, 3)
    ms_nmf_stream_w_kernel(const float* __restrict__ X, long long n, int m, const MsNmfProblem* __restrict__ problems,
                           float* __restrict__ Wg, const float* __restrict__ Hg, MsNmfStreamState* __restrict__ states) {
    extern __shared__ float sm[];
    const MsNmfProblem pb = problems[blockIdx.y];
    MsNmfStreamState* stt = states + blockIdx.y;
    if (stt->done) return;
    float* Wp = Wg + pb.w_off;
    const float* Hp = Hg + pb.h_off;
    const float* Xp = X + pb.x_off;
#define NMF_STREAM_W(KK) ms_nmf_stream_w_body<KK>(Xp, n, m, Wp, Hp, stt, sm)
    MS_NMF_K_SWITCH(pb.k, NMF_STREAM_W)
#undef NMF_STREAM_W
}

// mode 0: prepare (H H^T of the initial H, clear accumulators); mode 1: H update after a W pass
__global__ void __launch_bounds__(128)
    ms_nmf_stream_h_kernel(int m, const MsNmfProblem* __restrict__ problems, float* __restrict__ Hg,
                           MsNmfStreamState* __restrict__ states, const float* __restrict__ xx, int mode, int iteration,
                           float tol, int check_every) {
    __shared__ float sH[MS_NMF_MAX_K * MS_NMF_MAX_M];
    const MsNmfProblem pb = problems[blockIdx.x];
    MsNmfStreamState* stt = states + blockIdx.x;
    const int k = pb.k, tid = threadIdx.x;
    float* Hp = Hg + pb.h_off;
    if (mode == 1 && stt->done) return;
    if (mode == 0) {
        if (tid == 0) {
            stt->done = 0;
            stt->n_iter = 0;
            stt->err0 = stt->prev = stt->err = 0.f;
        }
        for (int e = tid; e < k * m; e += 128) sH[e] = Hp[e];
    } else {
        const float* WtW = stt->acc;
        const float* WtX = stt->acc + k * k;
        for (int e = tid; e < k * m; e += 128) {
            const int a = e / m, j = e % m;
            float den = 0.f;
            for (int b = 0; b < k; b++) den = fmaf(WtW[a * k + b], Hp[b * m + j], den);
            if (den == 0.f) den = NMF_EPS;
            sH[e] = Hp[e] * (WtX[e] / den);
        }
    }
    __syncthreads();
    if (mode == 1)
        for (int e = tid; e < k * m; e += 128) Hp[e] = sH[e];
    for (int e = tid; e < k * k; e += 128) {
        const int a = e / k, b = e % k;
        float acc = 0.f;
        for (int j = 0; j < m; j++) acc = fmaf(sH[a * m + j], sH[b * m + j], acc);
        stt->HHt[e] = acc;
    }
    __syncthreads();
    if (mode == 1) {
        // ||X - W H||^2 = ||X||^2 - 2 <H, W^T X> + <W^T W, H H^T>   (W^T X, W^T W of the updated W)
        double part = 0.0;
        for (int e = tid; e < k * m; e += 128) part -= 2.0 * (double)sH[e] * (double)stt->acc[k * k + e];
        for (int e = tid; e < k * k; e += 128) part += (double)stt->acc[e] * (double)stt->HHt[e];
        for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
        __shared__ double s_part[4];
        if ((tid & 31) == 0) s_part[tid >> 5] = part;
        __syncthreads();
        if (tid == 0) {
            const double sq = (double)xx[blockIdx.x] + s_part[0] + s_part[1] + s_part[2] + s_part[3];
            const float err = (float)sqrt(sq > 0.0 ? sq : 0.0);
            stt->err = err;
            stt->n_iter = iteration;
            if (iteration == 0) {
                stt->err0 = stt->prev = err;
            } else if (tol > 0.f && iteration % check_every == 0) {
                if (stt->err0 == 0.f || (stt->prev - err) / stt->err0 < tol) stt->done = 1;  // exact factorisation: converged
                stt->prev = err;
            }
        }
        __syncthreads();
    }
    for (int e = tid; e < k * k + k * m; e += 128) stt->acc[e] = 0.f;
}

// sum of squares of every column of X (per problem's X) and of the residual X - W H: VAF
__global__ void __launch_bounds__(256)
    ms_nmf_stream_vaf_kernel(const float* __restrict__ X, long long n, int m, const MsNmfProblem* __restrict__ problems,
                             const float* __restrict__ Wg, const float* __restrict__ Hg, double* __restrict__ sums) {
    // sums: [P][2][m]  (residual, total)
    __shared__ float sH[MS_NMF_MAX_K * MS_NMF_MAX_M];
    const MsNmfProblem pb = problems[blockIdx.y];
    const int k = pb.k;
    const float* Xp = X + pb.x_off;
    const float* Wp = Wg + pb.w_off;
    for (int e = threadIdx.x; e < k * m; e += 256) sH[e] = Hg[pb.h_off + e];
    __syncthreads();
    // thread -> column j = tid % m, rows strided: coalesced over the row-major X
    const int j = threadIdx.x % m, lane_row = threadIdx.x / m, rows_per_pass = 256 / m;
    if (lane_row >= rows_per_pass) return;
    double rs = 0.0, cs = 0.0;
    for (long long i = (long long)blockIdx.x * rows_per_pass + lane_row; i < n; i += (long long)gridDim.x * rows_per_pass) {
        float r = Xp[i * m + j];
        cs += (double)r * r;
        for (int c = 0; c < k; c++) r = fmaf(-Wp[i * k + c], sH[c * m + j], r);
        rs += (double)r * r;
    }
    atomicAdd(&sums[((long long)blockIdx.y * 2 + 0) * m + j], rs);
    atomicAdd(&sums[((long long)blockIdx.y * 2 + 1) * m + j], cs);
}

__global__ void ms_nmf_stream_finish_kernel(int m, const MsNmfStreamState* __restrict__ states,
                                            const double* __restrict__ sums, int32_t* __restrict__ n_iter,
                                            float* __restrict__ err, float* __restrict__ vaf, float* __restrict__ xx_out) {
    const int p = blockIdx.x;
    if (threadIdx.x == 0) {
        double rs = 0.0, cs = 0.0;
        for (int j = 0; j < m; j++) {
            rs += sums[((long long)p * 2 + 0) * m + j];
            cs += sums[((long long)p * 2 + 1) * m + j];
        }
        if (vaf) {
            vaf[(long long)p * (m + 1)] = (float)(1.0 - rs / cs);
            for (int j = 0; j < m; j++)
                vaf[(long long)p * (m + 1) + 1 + j] =
                    (float)(1.0 - sums[((long long)p * 2 + 0) * m + j] / sums[((long long)p * 2 + 1) * m + j]);
            n_iter[p] = states[p].n_iter;
            err[p] = (float)sqrt(rs);
        }
        if (xx_out) xx_out[p] = (float)cs;
    }
}

__global__ void ms_nmf_stream_err0_kernel(int m, MsNmfStreamState* __restrict__ states, const double* __restrict__ sums) {
    const int p = blockIdx.x;
    if (threadIdx.x == 0) {
        double rs = 0.0;
        for (int j = 0; j < m; j++) rs += sums[((long long)p * 2 + 0) * m + j];
        states[p].err0 = states[p].prev = states[p].err = (float)sqrt(rs);
    }
}

extern "C" int64_t ms_nmf_stream_workspace_bytes(int32_t m, int32_t n_problems) {
    return (int64_t)n_problems * ((int64_t)sizeof(MsNmfProblem) + (int64_t)sizeof(MsNmfStreamState) + 2 * m * 8 + 16) + 256;
}

// Same contract as ms_nmf_mu_batched for X of any length (X and W stream from HBM every
// iteration).  d_work: ms_nmf_stream_workspace_bytes(m, n_problems).  Synchronises `stream`
// every 64 iterations when tol > 0 to stop once every problem has converged.
extern "C" int ms_nmf_mu_stream(const float* d_X, int64_t n, int32_t m, const int32_t* h_ranks, const int32_t* h_x_index,
                                int32_t n_problems, float* d_W, float* d_H, int32_t max_iter, float tol,
                                int32_t check_every, void* d_work, int32_t* d_n_iter, float* d_err, float* d_vaf,
                                void* stream) {
    if (!d_X || !h_ranks || !d_W || !d_H || !d_work || !d_n_iter || !d_err || !d_vaf) return MS_E_INVALID;
    if (n < 1 || m < 1 || m > MS_NMF_MAX_M || n_problems < 0 || max_iter < 0 || check_every < 1) return MS_E_INVALID;
    if (n_problems == 0) return MS_OK;
    cudaStream_t st = (cudaStream_t)stream;
    char* wsp = (char*)d_work;
    MsNmfProblem* d_problems = (MsNmfProblem*)wsp;
    wsp += ms_align256(sizeof(MsNmfProblem) * n_problems);
    MsNmfStreamState* d_states = (MsNmfStreamState*)wsp;
    wsp += ms_align256(sizeof(MsNmfStreamState) * n_problems);
    double* d_sums = (double*)wsp;
    wsp += (size_t)n_problems * 2 * m * 8;
    float* d_xx = (float*)wsp;
    const int kmax = ms_nmf_upload_table(n, m, h_ranks, h_x_index, n_problems, d_problems, st);
    if (kmax < 0) return kmax;

    const long long n_tiles = (n + NMFS_ROWS - 1) / NMFS_ROWS;
    int ctas = (148 * 3 + n_problems - 1) / n_problems;  // three CTAs of the W pass fit an SM: one wave
    if (ctas > n_tiles) ctas = (int)n_tiles;
    if (ctas < 1) ctas = 1;
    const int KPmax = ms_nmf_pad4(kmax), MPs = ms_nmf_pad4(m);
    const size_t smem = sizeof(float) * (2 * (size_t)NMFS_ROWS * ms_nmf_stride(MPs) + 2 * (size_t)NMFS_ROWS * ms_nmf_stride(KPmax) +
                                         (size_t)MPs * KPmax + (size_t)kmax * KPmax);  // two tile buffers
    MS_CUDA_CHECK(cudaFuncSetAttribute(ms_nmf_stream_w_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    long long vaf_want = 148 * 8 / (n_problems < 8 ? n_problems : 8) + 1, vaf_cap = (long long)((n + 15) / 16);
    int vaf_ctas = (int)(vaf_want < vaf_cap ? vaf_want : vaf_cap);

    // ||X||^2 per problem (for the objective), then the objective of the initial factors
    MS_CUDA_CHECK(cudaMemsetAsync(d_sums, 0, (size_t)n_problems * 2 * m * 8, st));
    ms_nmf_stream_vaf_kernel<<<dim3(vaf_ctas, n_problems), 256, 0, st>>>(d_X, n, m, d_problems, d_W, d_H, d_sums);
    MS_COUNT_LAUNCH();
    ms_nmf_stream_finish_kernel<<<n_problems, 32, 0, st>>>(m, d_states, d_sums, nullptr, nullptr, nullptr, d_xx);
    MS_COUNT_LAUNCH();
    ms_nmf_stream_h_kernel<<<n_problems, 128, 0, st>>>(m, d_problems, d_H, d_states, d_xx, 0, 0, tol, check_every);
    MS_COUNT_LAUNCH();
    // error_at_init: the residual sums just computed are those of (W0, H0)
    ms_nmf_stream_err0_kernel<<<n_problems, 32, 0, st>>>(m, d_states, d_sums);
    MS_COUNT_LAUNCH();

    for (int it = 1; it <= max_iter; it++) {
        ms_nmf_stream_w_kernel<<<dim3(ctas, n_problems), NMFS_ROWS, smem, st>>>(d_X, n, m, d_problems, d_W, d_H, d_states);
        MS_COUNT_LAUNCH();
        ms_nmf_stream_h_kernel<<<n_problems, 128, 0, st>>>(m, d_problems, d_H, d_states, d_xx, 1, it, tol, check_every);
        MS_COUNT_LAUNCH();
        if (tol > 0.f && it % 64 == 0) {  // stop early when every problem has converged
            const int done = ms_nmf_all_done(d_states, n_problems, st);
            if (done < 0) return done;
            if (done) break;
        }
    }
    MS_CUDA_CHECK(cudaMemsetAsync(d_sums, 0, (size_t)n_problems * 2 * m * 8, st));
    ms_nmf_stream_vaf_kernel<<<dim3(vaf_ctas, n_problems), 256, 0, st>>>(d_X, n, m, d_problems, d_W, d_H, d_sums);
    MS_COUNT_LAUNCH();
    ms_nmf_stream_finish_kernel<<<n_problems, 32, 0, st>>>(m, d_states, d_sums, d_n_iter, d_err, d_vaf, nullptr);
    MS_COUNT_LAUNCH();
    MS_CUDA_CHECK(cudaGetLastError());
    return MS_OK;
}
