// K2: (multi-class) Bayesian logistic regression -- ELBO forward + pathwise backward in ONE pass over X.
// See include/brancher_cuda.h (brn_linear_elbo_fwd_bwd).
//
// "Columns" j = (sample s, class c): Wmat [J = S*C, F].  A CTA owns one tile of 128 columns (whole
// samples only) and walks a contiguous group of 128-row tiles of X:
//   phase 1   L[128 rows, 128 cols]   = Xtile . Wtile^T                       (K = F)
//   phase 2   ll += log-lik(L, y) ; dL = d ll / d L                            (registers / smem)
//   phase 3   dWacc[128 cols, F]     += dL^T . Xtile                           (K = 128 rows)
// dWacc lives in registers for the CTA's whole row group and is flushed once with atomics, so X is read
// from HBM once per column tile (and those re-reads are L2 hits: column tiles of one row group are
// scheduled together) and nothing of size S x N ever reaches memory.
#include "meanfield.cuh"
#include "umma_gemm.cuh"
#include <optional>
#include <stdlib.h>

namespace brn {

constexpr int LN_T = 128;            // tile edge (rows, columns, max features)
constexpr int LN_LD = LN_T + 4;      // smem leading dimension (keeps float4 alignment)

// Likelihood codes of brn_linear_* (include/brancher_cuda.h); brn_linreg_* continue them with BRN_LINREG_NORMAL / _CAUCHY /
// _LAPLACE.  The LIK template argument of linear_fused_kernel and linear_flash_kernel takes these codes.
constexpr int LIN_BERNOULLI = 0, LIN_CATEGORICAL = 1;

struct LinearArgs {
    const float* X; const void* y; int64_t N; int F, C, S;
    const float* W; float* dW;       // [S*C, F] contiguous
    int tiles_per_group; int64_t n_row_tiles;
    float inv_S; double* loss;
    double* ll_cols;                 // optional [S]: per-sample log-likelihood sums (K6), += ; loss may then be NULL
    const float* sigma;              // LIK == 3: [S] noise scale per sample
    double* ll_cols2;                // LIK == 3: [S] += sum z^2 / (1 + z^2)
};

// LIK, the likelihood code of the C ABI: 0: Bernoulli/Binomial(1) with float y, 1: Categorical with int32 labels, 2: Gaussian
// residuals with float y (C == 1): d = r = y - l and ll_cols[s] += sum r^2 (loss unused; the noise scale is applied per sample
// afterwards, linreg_finish_kernel),
// 3: Cauchy residuals (C == 1): z = r / sigma_s, d = z / (1 + z^2), ll_cols[s] += sum log1p(z^2), ll_cols2[s] += sum z^2/(1 + z^2),
// 4: Laplace residuals (C == 1): d = sign(r), ll_cols[s] += sum |r|  (3, 4: loss unused, finished by linreg_finish_kernel)
template <int LIK>
__global__ void __launch_bounds__(256, 1) linear_fused_kernel(LinearArgs a) {
    extern __shared__ __align__(16) float sm[];
    float (*Xs)[LN_LD] = reinterpret_cast<float (*)[LN_LD]>(sm);                       // [row][f]
    float (*Ws)[LN_LD] = reinterpret_cast<float (*)[LN_LD]>(sm + LN_T * LN_LD);        // [f][col]
    float (*Ls)[LN_LD] = reinterpret_cast<float (*)[LN_LD]>(sm + 2 * LN_T * LN_LD);    // [row][col]
    float* ys = sm + 3 * LN_T * LN_LD;                                                 // [row] (bit-cast for labels)
    __shared__ double red[32];

    const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
    const int F = a.F, C = a.C;
    const int spc = LN_T / C;                 // whole samples per column tile
    const int ncols = spc * C;
    const int s_base = blockIdx.x * spc;
    const int64_t J = (int64_t)a.S * C, j0 = (int64_t)s_base * C;
    const bool xvec = (F % 4 == 0) && ((uintptr_t)a.X % 16 == 0);

    // W tile, transposed to [f][col]; zero outside
    for (int idx = t; idx < LN_T * LN_T; idx += 256) {
        int col = idx >> 7, f = idx & 127;
        float v = 0.f;
        if (col < ncols && j0 + col < J && f < F) v = a.W[(j0 + col) * F + f];
        Ws[f][col] = v;
    }

    float acc2[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc2[i][j] = 0.f;
    double ll_thread = 0.0;
    double llc[8];                   // LIK == 0 / 2 with ll_cols: this thread's 8 columns, summed over its rows and tiles
#pragma unroll
    for (int j = 0; j < 8; ++j) llc[j] = 0.0;
    __shared__ double llcol_s[LN_T];  // LIK == 1 with ll_cols: per sample of the tile; LIK == 3: sum z^2 / (1 + z^2) per column
    if (a.ll_cols && t < LN_T) llcol_s[t] = 0.0;
    float isg[8];                    // LIK == 3: 1 / sigma of this thread's 8 columns
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        isg[j] = 1.f;
        if (LIK == BRN_LINREG_CAUCHY) {
            const int col = (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
            if (col < ncols && j0 + col < J) isg[j] = 1.f / a.sigma[j0 + col];
        }
    }

    const int64_t tile_begin = (int64_t)blockIdx.y * a.tiles_per_group;
    const int64_t tile_end = min(a.n_row_tiles, tile_begin + a.tiles_per_group);
    for (int64_t tile = tile_begin; tile < tile_end; ++tile) {
        const int64_t r0 = tile * LN_T;
        __syncthreads();   // previous tile's phase 3 done with Xs / Ls
        // ---- load X tile [128][F] (zero padded to 128 features / N rows)
        if (xvec) {
            for (int idx = t; idx < LN_T * (LN_T / 4); idx += 256) {
                int row = idx >> 5, f4 = (idx & 31) * 4;
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (r0 + row < a.N && f4 < F) v = *reinterpret_cast<const float4*>(a.X + (r0 + row) * F + f4);
                *reinterpret_cast<float4*>(&Xs[row][f4]) = v;
            }
        } else {
            for (int idx = t; idx < LN_T * LN_T; idx += 256) {
                int row = idx >> 7, f = idx & 127;
                Xs[row][f] = (r0 + row < a.N && f < F) ? a.X[(r0 + row) * F + f] : 0.f;
            }
        }
        if (t < LN_T) {
            float v = 0.f;
            if (r0 + t < a.N) {
                if (LIK != LIN_CATEGORICAL) v = reinterpret_cast<const float*>(a.y)[r0 + t];
                else v = __int_as_float(reinterpret_cast<const int32_t*>(a.y)[r0 + t]);
            }
            ys[t] = v;
        }
        __syncthreads();

        // ---- phase 1: logits
        float acc[8][8];
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
        const int k4n = (F + 3) >> 2;
        for (int k4 = 0; k4 < k4n; ++k4) {
            float4 xa[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                int row = (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
                xa[i] = *reinterpret_cast<const float4*>(&Xs[row][k4 * 4]);
            }
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                float4 b0 = *reinterpret_cast<const float4*>(&Ws[k4 * 4 + kk][tx * 4]);
                float4 b1 = *reinterpret_cast<const float4*>(&Ws[k4 * 4 + kk][64 + tx * 4]);
                float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    float av = kk == 0 ? xa[i].x : kk == 1 ? xa[i].y : kk == 2 ? xa[i].z : xa[i].w;
#pragma unroll
                    for (int j = 0; j < 8; ++j) acc[i][j] = __fmaf_rn(av, bv[j], acc[i][j]);
                }
            }
        }

        // ---- phase 2: log-likelihood and d ll / d logit
        float ll_tile = 0.f;
        if (LIK != LIN_CATEGORICAL) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                int row = (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
                bool rv = r0 + row < a.N;
                float yv = ys[row];
                float d[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    int col = (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
                    bool ok = rv && col < ncols && (j0 + col) < J;
                    if constexpr (LIK == BRN_LINREG_NORMAL) {
                        d[j] = ok ? yv - acc[i][j] : 0.f;
                        if (a.ll_cols) llc[j] += (double)(d[j] * d[j]);
                    } else if constexpr (LIK == BRN_LINREG_CAUCHY) {
                        const float r = ok ? yv - acc[i][j] : 0.f;
                        const float z = r * isg[j], z2 = z * z, iq = 1.f / (1.f + z2);
                        d[j] = z * iq;
                        llc[j] += (double)log1pf(z2);
                        if (z2 != 0.f) atomicAdd(&llcol_s[col], (double)(z2 * iq));      // sixteen threads share a column
                    } else if constexpr (LIK == BRN_LINREG_LAPLACE) {
                        const float r = ok ? yv - acc[i][j] : 0.f;
                        d[j] = r > 0.f ? 1.f : (r < 0.f ? -1.f : 0.f);      // sign(0) = 0, as torch's abs gradient
                        llc[j] += (double)fabsf(r);
                    } else {
                        float l = acc[i][j];
                        float sp = log1pexpf(l);
                        const float lv = ok ? __fmaf_rn(yv, l, -sp) : 0.f;
                        ll_tile += lv;
                        if (a.ll_cols) llc[j] += (double)lv;
                        d[j] = ok ? yv - sigmoidf(l) : 0.f;
                    }
                }
                *reinterpret_cast<float4*>(&Ls[row][tx * 4]) = make_float4(d[0], d[1], d[2], d[3]);
                *reinterpret_cast<float4*>(&Ls[row][64 + tx * 4]) = make_float4(d[4], d[5], d[6], d[7]);
            }
            __syncthreads();
        } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                int row = (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
                *reinterpret_cast<float4*>(&Ls[row][tx * 4]) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
                *reinterpret_cast<float4*>(&Ls[row][64 + tx * 4]) = make_float4(acc[i][4], acc[i][5], acc[i][6], acc[i][7]);
            }
            __syncthreads();
            for (int item = t; item < LN_T * spc; item += 256) {
                int sl = item % spc, row = item / spc;
                float* lg = &Ls[row][sl * C];
                bool ok = (r0 + row < a.N) && (s_base + sl < a.S);
                if (!ok) {
                    for (int c = 0; c < C; ++c) lg[c] = 0.f;
                    continue;
                }
                int label = __float_as_int(ys[row]);
                float m = -INFINITY;
                for (int c = 0; c < C; ++c) m = fmaxf(m, lg[c]);
                float se = 0.f;
                for (int c = 0; c < C; ++c) se += expf(lg[c] - m);
                float lse = m + logf(se);
                for (int c = 0; c < C; ++c) {
                    float l = lg[c];
                    if (c == label) {
                        ll_tile += l - lse;
                        if (a.ll_cols) atomicAdd(&llcol_s[sl], (double)(l - lse));
                    }
                    lg[c] = (c == label ? 1.f : 0.f) - expf(l - lse);
                }
            }
            // columns beyond ncols (tile padding) must not contribute to phase 3
            if (ncols < LN_T)
                for (int idx = t; idx < LN_T * (LN_T - ncols); idx += 256) {
                    int row = idx / (LN_T - ncols), col = ncols + idx % (LN_T - ncols);
                    Ls[row][col] = 0.f;
                }
            __syncthreads();
        }
        ll_thread += (double)ll_tile;

        // ---- phase 3: dW[col, f] += sum_row dL[row, col] * X[row, f]   (skipped when only the log-likelihoods are wanted)
        if (a.dW == nullptr) continue;
#pragma unroll 4
        for (int row = 0; row < LN_T; ++row) {
            float4 a0 = *reinterpret_cast<const float4*>(&Ls[row][ty * 4]);
            float4 a1 = *reinterpret_cast<const float4*>(&Ls[row][64 + ty * 4]);
            float4 b0 = *reinterpret_cast<const float4*>(&Xs[row][tx * 4]);
            float4 b1 = *reinterpret_cast<const float4*>(&Xs[row][64 + tx * 4]);
            float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc2[i][j] = __fmaf_rn(av[i], bv[j], acc2[i][j]);
        }
    }

    // ---- flush
    if (a.ll_cols) {
        if (LIK != LIN_CATEGORICAL) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int col = (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
                if (col < ncols && j0 + col < J && llc[j] != 0.0) atomicAdd(&a.ll_cols[j0 + col], llc[j]);
            }
            if (LIK == BRN_LINREG_CAUCHY) {
                __syncthreads();
                if (t < ncols && j0 + t < J && llcol_s[t] != 0.0) atomicAdd(&a.ll_cols2[j0 + t], llcol_s[t]);
            }
        } else {
            __syncthreads();
            if (t < spc && s_base + t < a.S && llcol_s[t] != 0.0) atomicAdd(&a.ll_cols[s_base + t], llcol_s[t]);
        }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        if (a.dW == nullptr) break;
        int col = (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
        if (col >= ncols || j0 + col >= J) continue;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            int f = (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
            if (f < F) atomicAdd(&a.dW[(j0 + col) * F + f], acc2[i][j]);
        }
    }
    double tot = block_sum<double>(ll_thread, red);
    if (t == 0 && a.loss) atomicAdd(a.loss, -tot * (double)a.inv_S);
}

constexpr int LT_BN1 = 256;       // logits GEMM: samples per n-tile (16 epilogue warps x 64 columns)
constexpr int LT_EW1 = 16;
constexpr int LT_BN2 = 128;       // gradient GEMM: features per n-tile (F <= 128)
constexpr int LT_BK = 16;
constexpr int LT_BK2 = 32;        // gradient GEMM: 128-byte operand rows (both operands are scattered K-major rows: half the requests)

// rows per chunk of the tcgen05 path: whole 128-row tiles such that (m-tiles x n-tiles) fills ~2 rounds of the grid
static int linear_tc_chunk_rows(int S, int sms) {
    const int n_tiles = (S + LT_BN1 - 1) / LT_BN1;
    const int rounds = 12;     // measured at C2 on B200 (profiles/r1k_*, r1l_*): 2: 7.06 ms, 4: 5.90, 8: 5.43, 12: 5.14, 16: 5.19, 24: 5.14
    int mt = rounds * sms / n_tiles;
    if (mt < 1) mt = 1;
    if (mt > 512) mt = 512;
    return mt * 128;
}

// dW[i] = sum_j part[j * stride + i]
__global__ void sum_slices_kernel(const float* __restrict__ part, int slices, int64_t stride, int64_t n, float* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float acc = 0.f;
    for (int j = 0; j < slices; ++j) acc += part[(int64_t)j * stride + i];
    out[i] = acc;
}

}  // namespace brn
#include "linear_flash.cuh"
namespace brn {

static int check_prepared_x(const char* fn, const void* px, int64_t N, int F) {
    BRN_CHECK_ARG(!px || (linear_prepared_x_bytes(N, F) > 0 && (reinterpret_cast<uintptr_t>(px) & 255) == 0),
                  "%s: a prepared X does not exist for N=%lld F=%d, or px is not 256-byte aligned", fn, (long long)N, F);
    return 0;
}

// TF32-split operands and scratch of the tcgen05 variant (Bernoulli, C == 1); S = weight vectors (MC samples or particles)
struct LinearTcBuffers {
    LinearFlashBuffers flash;
    float *Wh, *Wl, *Xh, *Xl, *Xth, *Xtl, *dT, *dWpart;
    int64_t ldF, ldN, ldNB, n_chunks;
    int nb, slices;
    template <class Take>
    void carve(Take&& take, int S, int64_t N, int F, int sms) {
        ldF = (F + 3) / 4 * 4;
        ldN = (N + 3) / 4 * 4;
        nb = linear_tc_chunk_rows(S, sms);
        if (nb > N) nb = (int)((N + 127) / 128 * 128);
        ldNB = nb;
        const int m2 = (S + UG_BM - 1) / UG_BM;
        slices = (2 * m2 <= sms) ? sms / m2 : 1;
        Wh = take((size_t)S * ldF); Wl = take((size_t)S * ldF);
        Xh = take((size_t)N * ldF); Xl = take((size_t)N * ldF);
        // X^T is stored PER ROW CHUNK, [chunk][F][nb]: the 128 feature rows of a gradient-GEMM B tile are then nb*4 bytes
        // apart (one or two MB in total) instead of N*4 bytes (4 MB pitch at N = 10^6: 128 rows = 128 different 2 MB pages
        // per TMA request -- measured: the gradient GEMM spent 71 % of its time waiting for those loads)
        n_chunks = nb > 0 ? (N + nb - 1) / nb : 0;
        Xth = take((size_t)n_chunks * F * ldNB); Xtl = take((size_t)n_chunks * F * ldNB);
        dT = take((size_t)S * ldNB);
        dWpart = take((size_t)slices * S * F);
        flash.carve(take, S, F, sms);
        flash.Xh = reinterpret_cast<__half*>(Xh);        // the one-pass kernel's fp16 pair of X lives in the staged pair's buffers
        flash.Xl = reinterpret_cast<__half*>(Xl);
    }
};

struct LinearWorkspace {
    float *eps, *W, *dW, *stats;
    LinearTcBuffers tc;
    size_t bytes;
    LinearWorkspace(void* base, int64_t numel, int S, int64_t N, int F, bool use_tc, int sms) {
        WorkspaceCarver take(base);
        eps = take((size_t)S * numel);
        W = take((size_t)S * numel);
        dW = take((size_t)S * numel);
        stats = take(4 * (size_t)((numel + 3) / 4 * 4));
        tc = LinearTcBuffers();
        if (use_tc) tc.carve(take, S, N, F, sms);
        bytes = take.off;
    }
};

// particles: G = -(d ll / d theta) - d log N(theta; a, b) / d theta ; loss += sum -log N(theta; a, b)
__global__ void __launch_bounds__(256)
particles_prior_kernel(const float* __restrict__ theta, const float* __restrict__ prior_loc, const float* __restrict__ prior_scale,
                       int64_t numel, int64_t total, float* __restrict__ G, double* __restrict__ loss) {
    __shared__ double red[32];
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double nlp = 0.0;
    if (i < total) {
        float g = -G[i];
        if (prior_loc) {
            const int64_t e = i % numel;
            const float a = prior_loc[e], b = prior_scale[e], df = theta[i] - a, inv_b2 = 1.0f / (b * b);
            g = __fmaf_rn(df, inv_b2, g);
            nlp = (double)(0.5f * df * df * inv_b2 + logf(b) + BRN_HALF_LOG_2PI);
        }
        G[i] = g;
    }
    double tot = block_sum<double>(nlp, red);
    if (threadIdx.x == 0 && prior_loc) atomicAdd(loss, tot);
}

// the shapes the staged tcgen05 pair takes (with the Bernoulli likelihood): what BRN_LINEAR_VARIANT=tcgen05 forces, and what
// the workspace is sized for
static bool linear_tc_shape(int64_t N, int F, int C, int S) { return C == 1 && F % 4 == 0 && F <= LT_BN2 && N >= 1 && S >= 1; }

static bool linear_use_tc(int likelihood, int64_t N, int F, int C, int S) {
    bool tc = likelihood == LIN_BERNOULLI && linear_tc_shape(N, F, C, S) && N >= 4096 && S >= 64;
    if (const char* env = getenv("BRN_LINEAR_VARIANT")) {
        if (!strcmp(env, "simt")) tc = false;
        else if (!strcmp(env, "tcgen05")) tc = likelihood == LIN_BERNOULLI && linear_tc_shape(N, F, C, S);
    }
    return tc;
}

}  // namespace brn

using namespace brn;

static int launch_linear_fused(const float* X, const void* y, int likelihood, int64_t N, int F, int C, int S, const float* W,
                               float* dW, float inv_S, double* loss, cudaStream_t stream, double* ll_cols = nullptr,
                               const float* sigma = nullptr, double* ll_cols2 = nullptr) {
    LinearArgs a;
    a.X = X; a.y = y; a.N = N; a.F = F; a.C = C; a.S = S; a.W = W; a.dW = dW;
    a.inv_S = inv_S; a.loss = loss; a.ll_cols = ll_cols; a.sigma = sigma; a.ll_cols2 = ll_cols2;
    const int spc = LN_T / C;
    const int col_tiles = (S + spc - 1) / spc;
    a.n_row_tiles = (N + LN_T - 1) / LN_T;
    int64_t groups = device_sm_count() / col_tiles;
    if (groups < 1) groups = 1;
    if (groups > a.n_row_tiles) groups = a.n_row_tiles;
    a.tiles_per_group = (int)((a.n_row_tiles + groups - 1) / groups);
    groups = (a.n_row_tiles + a.tiles_per_group - 1) / a.tiles_per_group;
    const size_t smem = sizeof(float) * (3 * LN_T * LN_LD + LN_T);
    dim3 grid(col_tiles, (unsigned)groups);
    auto launch = [&](auto kern) -> int {
        BRN_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<grid, 256, smem, stream>>>(a);
        return 0;
    };
    int e;
    if (likelihood == LIN_BERNOULLI) e = launch(linear_fused_kernel<LIN_BERNOULLI>);
    else if (likelihood == BRN_LINREG_NORMAL) e = launch(linear_fused_kernel<BRN_LINREG_NORMAL>);
    else if (likelihood == BRN_LINREG_CAUCHY) e = launch(linear_fused_kernel<BRN_LINREG_CAUCHY>);
    else if (likelihood == BRN_LINREG_LAPLACE) e = launch(linear_fused_kernel<BRN_LINREG_LAPLACE>);
    else e = launch(linear_fused_kernel<LIN_CATEGORICAL>);
    if (e) return e;
    BRN_LAUNCH_OK("linear_fused_kernel");
    return 0;
}

// tcgen05 variant of the fused Bernoulli log-likelihood + gradient for S weight vectors W [S, F] (N > 0):
//   per row chunk, (1) logits GEMM with the Bernoulli likelihood fused in its epilogue (writes d = y - sigmoid(l)
//   transposed + TF32-split; loss += loss_scale * sum ll), (2) gradient GEMM dW[s,f] += d^T X, K-split over the grid
//   with per-slice accumulation (no atomics); finally the slices are summed into dW [S, F] = + d ll / d W.
static int launch_linear_tc(const float* X, const float* y, int64_t N, int F, int S, const float* W, float* dW, float loss_scale,
                            double* loss, const LinearTcBuffers& b, const char* stage_split, const char* stage_fused,
                            cudaStream_t stream, const void* px = nullptr) {
    if (linear_flash_ok(X, N, F, S)) {
        // one pass over X: logits MMA -> likelihood -> d through shared memory -> gradient MMA (linear_flash.cuh)
        set_variant("tcgen05-flash");
        StageTimer st2(stage_fused, stream);
        return launch_linear_flash(LIN_BERNOULLI, X, px, y, N, F, S, W, dW, loss_scale, loss, nullptr, nullptr, nullptr, b.flash,
                                   stream);
    }
    constexpr int drain = 2;
    // Operands that cross HBM once are kept as ONE fp32 matrix and split into TF32 (hi, lo) inside the GEMMs by converter warps
    // (SPLIT mask, umma_gemm.cuh): d^T between the two GEMMs, and X itself (read in place: no row-major copy at all) when
    // TMA can read it (16-byte aligned base); the per-chunk X^T stays pre-split.  Measured at C2 on B200 (profiles/r1t_*,
    // mask of plain operands 1 = d^T, 2 = X^T, 4 = X): 0: 5.44 ms, 1: 4.75, 3: 5.07, 5: 4.57, 7: 4.69 -- converting the B
    // tile too slows the gradient GEMM more than the smaller split pass saves
    const bool x_in_place = reinterpret_cast<uintptr_t>(X) % 16 == 0;
    {
        StageTimer sp(stage_split, stream);
        if (int e = launch_split_tf32(W, F, S, F, b.Wh, b.Wl, b.ldF, nullptr, nullptr, 0, stream)) return e;
        for (int64_t c = 0; c < b.n_chunks; ++c) {
            const int64_t r0 = c * b.nb;
            const int nb = (int)((N - r0 < b.nb) ? (N - r0) : b.nb);
            // (hi, lo) of X transposed and, unless X is read in place, row-major; an unused output pair is skipped by the kernel
            if (int e = launch_split_tf32(X + r0 * F, F, nb, F, x_in_place ? nullptr : b.Xh + r0 * b.ldF,
                                          x_in_place ? nullptr : b.Xl + r0 * b.ldF, b.ldF, b.Xth + c * F * b.ldNB,
                                          b.Xtl + c * F * b.ldNB, b.ldNB, stream))
                return e;
        }
        BRN_CUDA_OK(cudaMemsetAsync(b.dWpart, 0, sizeof(float) * (size_t)b.slices * S * F, stream));
    }
    StageTimer st2(stage_fused, stream);
    for (int64_t r0 = 0; r0 < N; r0 += b.nb) {
        const int nb = (int)((N - r0 < b.nb) ? (N - r0) : b.nb);
        EpiBernoulli::Params e1;
        e1.y = y + r0; e1.dT = b.dT; e1.rows = nb; e1.cols = S;
        e1.ld = b.ldNB; e1.loss = loss; e1.neg_inv_S = loss_scale;
        if (x_in_place) {
            if (int e = launch_umma_nt<LT_BN1, LT_BK, EpiBernoulli, LT_EW1, 1, 2>(X + r0 * F, nullptr, nb, F, b.Wh, b.Wl, S, b.ldF, F, 0,
                                                                                   drain, e1, stream))
                return e;
        } else if (int e = launch_umma_nt<LT_BN1, LT_BK, EpiBernoulli, LT_EW1>(b.Xh + r0 * b.ldF, b.Xl + r0 * b.ldF, nb, b.ldF, b.Wh,
                                                                                b.Wl, S, b.ldF, F, 0, drain, e1, stream))
            return e;
        // K tail of the last chunk: the TMA box zero-fills columns >= nb of d^T (tensor map extent = nb)
        EpiAccum::Params e2;
        e2.out = b.dWpart; e2.rows = S; e2.cols = F; e2.ld = F; e2.slice_stride = (int64_t)S * F;
        const int64_t xt = (r0 / b.nb) * F * b.ldNB;
        if (int e = launch_umma_nt<LT_BN2, LT_BK2, EpiAccum, UG_EPI_WARPS, 1>(b.dT, nullptr, S, b.ldNB, b.Xth + xt, b.Xtl + xt, F, b.ldNB,
                                                                               nb, 0, drain, e2, stream, b.slices > 1))
            return e;
    }
    const int64_t tot = (int64_t)S * F;
    sum_slices_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, stream>>>(b.dWpart, b.slices, tot, tot, dW);
    BRN_LAUNCH_OK("sum_slices_kernel");
    return 0;
}

extern "C" size_t brn_linear_particles_workspace_bytes(int64_t N, int F, int C, int n) {
    if (N < 0 || F <= 0 || C <= 0 || n < 0) return 0;
    if (!linear_tc_shape(N, F, C, n)) return 0;      // only the tcgen05 variant needs scratch
    WorkspaceCarver take(nullptr);
    LinearTcBuffers b;
    b.carve(take, n, N, F, device_sm_count());
    return take.off;
}

extern "C" int brn_linear_particles_loss_grad(const float* X, const void* y, int likelihood, int64_t N, int F, int C,
                                              const float* theta, int n, const float* prior_loc, const float* prior_scale,
                                              float* G, double* loss, void* workspace, size_t workspace_bytes, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    BRN_CHECK_ARG(theta && G && loss, "brn_linear_particles_loss_grad: NULL pointer");
    BRN_CHECK_ARG(N >= 0 && F > 0 && C > 0 && n >= 0, "brn_linear_particles_loss_grad: bad shape N=%lld F=%d C=%d n=%d",
                  (long long)N, F, C, n);
    BRN_CHECK_ARG(N == 0 || (X && y), "brn_linear_particles_loss_grad: NULL data pointer");
    BRN_CHECK_ARG(F <= LN_T && C <= LN_T, "brn_linear_particles_loss_grad: F=%d / C=%d exceed the supported maximum %d", F, C, LN_T);
    BRN_CHECK_ARG(likelihood == LIN_BERNOULLI || likelihood == LIN_CATEGORICAL, "brn_linear_particles_loss_grad: unknown likelihood %d",
                  likelihood);
    BRN_CHECK_ARG(likelihood == LIN_CATEGORICAL || C == 1, "Bernoulli/Binomial likelihood needs C == 1 (got %d)", C);
    BRN_CHECK_ARG((prior_loc == nullptr) == (prior_scale == nullptr), "prior_loc and prior_scale must both be given or both NULL");
    if (n == 0) return 0;
    // tcgen05 variant (the K2 GEMM pair with the particles as the weight vectors) when the caller provides scratch
    const bool use_tc = workspace != nullptr && N > 0 && linear_use_tc(likelihood, N, F, C, n);
    set_variant(use_tc ? "tcgen05" : "simt");
    const int64_t numel = (int64_t)C * F, total = numel * n;
    if (use_tc) {
        WorkspaceCarver take(workspace);
        LinearTcBuffers b;
        b.carve(take, n, N, F, device_sm_count());
        BRN_CHECK_ARG(workspace_bytes >= take.off, "workspace too small: %zu < %zu", workspace_bytes, take.off);
        if (int e = launch_linear_tc(X, reinterpret_cast<const float*>(y), N, F, n, theta, G, -1.0f, loss, b,
                                     "particles.split_operands", "particles.loglik_grad", stream))
            return e;
    } else {
        BRN_CUDA_OK(cudaMemsetAsync(G, 0, sizeof(float) * (size_t)total, stream));
        if (N > 0) {
            StageTimer st("particles.loglik_grad", stream);
            if (int e = launch_linear_fused(X, y, likelihood, N, F, C, n, theta, G, 1.0f, loss, stream)) return e;
        }
    }
    StageTimer st2("particles.prior", stream);
    particles_prior_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(theta, prior_loc, prior_scale, numel, total, G, loss);
    BRN_LAUNCH_OK("particles_prior_kernel");
    return 0;
}

// K6 (b): per-vector log-likelihoods (and optionally their gradients) of n weight vectors, one fused pass over X
extern "C" int brn_linear_vectors_loglik_grad(const float* X, const void* y, int likelihood, int64_t N, int F, int C,
                                              const float* V, int n, float* G, double* ll, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    BRN_CHECK_ARG(V && ll, "brn_linear_vectors_loglik_grad: NULL pointer");
    BRN_CHECK_ARG(N >= 0 && F > 0 && C > 0 && n >= 0, "brn_linear_vectors_loglik_grad: bad shape N=%lld F=%d C=%d n=%d",
                  (long long)N, F, C, n);
    BRN_CHECK_ARG(N == 0 || (X && y), "brn_linear_vectors_loglik_grad: NULL data pointer");
    BRN_CHECK_ARG(F <= LN_T && C <= LN_T, "brn_linear_vectors_loglik_grad: F=%d / C=%d exceed the supported maximum %d", F, C, LN_T);
    BRN_CHECK_ARG(likelihood == LIN_BERNOULLI || likelihood == LIN_CATEGORICAL, "brn_linear_vectors_loglik_grad: unknown likelihood %d",
                  likelihood);
    BRN_CHECK_ARG(likelihood == LIN_CATEGORICAL || C == 1, "Bernoulli/Binomial likelihood needs C == 1 (got %d)", C);
    if (n == 0) return 0;
    set_variant("simt");
    const int64_t total = (int64_t)C * F * n;
    BRN_CUDA_OK(cudaMemsetAsync(ll, 0, sizeof(double) * (size_t)n, stream));
    if (G) BRN_CUDA_OK(cudaMemsetAsync(G, 0, sizeof(float) * (size_t)total, stream));
    if (N > 0) {
        StageTimer st("vectors.loglik_grad", stream);
        if (int e = launch_linear_fused(X, y, likelihood, N, F, C, n, V, G, 1.0f, nullptr, stream, ll)) return e;
        if (G) {       // the fused kernel accumulates +d ll / d V; the ABI returns the loss gradient -d ll / d V
            particles_prior_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(V, nullptr, nullptr, (int64_t)C * F, total, G,
                                                                                       nullptr);
            BRN_LAUNCH_OK("particles_prior_kernel");
        }
    }
    return 0;
}

extern "C" size_t brn_linear_workspace_bytes(int64_t N, int F, int C, int s_local) {
    if (N < 0 || F <= 0 || C <= 0 || s_local < 0) return 0;
    // sized for the larger of the two variants (the likelihood is not known here): tcgen05 buffers whenever C == 1
    return LinearWorkspace(nullptr, (int64_t)C * F, s_local, N, F, linear_tc_shape(N, F, C, s_local), device_sm_count()).bytes;
}

extern "C" size_t brn_linear_prepared_x_bytes(int64_t N, int F) { return linear_prepared_x_bytes(N, F); }

extern "C" int brn_linear_prepare_x(const float* X, int64_t N, int F, void* px, size_t px_bytes, void* stream_) {
    const size_t need = linear_prepared_x_bytes(N, F);
    BRN_CHECK_ARG(need > 0, "brn_linear_prepare_x: no prepared form for N=%lld F=%d (needs N >= 1, F a multiple of 16, F <= %d)", (long long)N, F,
                  LF_FMAX);
    BRN_CHECK_ARG(X && px && px_bytes >= need, "brn_linear_prepare_x: NULL pointer or buffer too small (%zu < %zu)", px_bytes, need);
    BRN_CHECK_ARG((reinterpret_cast<uintptr_t>(X) & 15) == 0 && (reinterpret_cast<uintptr_t>(px) & 255) == 0,
                  "brn_linear_prepare_x: X must be 16-byte and px 256-byte aligned");
    return launch_prepare_x(X, N, F, static_cast<float*>(px), prepared_x_hi(px), prepared_x_lo(px, N, F), (cudaStream_t)stream_);
}

extern "C" int brn_linear_elbo_fwd_bwd(const float* X, const void* y, int likelihood, int64_t N, int F, int C,
                                       const brn_mf_var* w, const brn_sample_range* r, void* workspace,
                                       size_t workspace_bytes, int with_prior, double* loss, void* stream_) {
    return brn_linear_elbo_fwd_bwd_px(X, nullptr, y, likelihood, N, F, C, w, r, workspace, workspace_bytes, with_prior, loss, stream_);
}

extern "C" int brn_linear_elbo_fwd_bwd_px(const float* X, const void* px, const void* y, int likelihood, int64_t N, int F, int C,
                                          const brn_mf_var* w, const brn_sample_range* r, void* workspace,
                                          size_t workspace_bytes, int with_prior, double* loss, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (int e = check_prepared_x("brn_linear_elbo_fwd_bwd_px", px, N, F)) return e;
    BRN_CHECK_ARG(w && r && loss, "brn_linear_elbo_fwd_bwd: NULL pointer");
    BRN_CHECK_ARG(N >= 0 && F > 0 && C > 0, "brn_linear_elbo_fwd_bwd: bad shape N=%lld F=%d C=%d", (long long)N, F, C);
    BRN_CHECK_ARG(N == 0 || (X && y), "brn_linear_elbo_fwd_bwd: NULL data pointer");
    BRN_CHECK_ARG(F <= LN_T, "brn_linear_elbo_fwd_bwd: F=%d exceeds the supported maximum %d", F, LN_T);
    BRN_CHECK_ARG(C <= LN_T, "brn_linear_elbo_fwd_bwd: C=%d exceeds the supported maximum %d", C, LN_T);
    BRN_CHECK_ARG(likelihood == LIN_BERNOULLI || likelihood == LIN_CATEGORICAL, "brn_linear_elbo_fwd_bwd: unknown likelihood %d", likelihood);
    BRN_CHECK_ARG(likelihood == LIN_CATEGORICAL || C == 1, "Bernoulli/Binomial likelihood needs C == 1 (got %d)", C);
    if (int e = check_sample_range(*r)) return e;
    const int64_t numel = (int64_t)C * F;
    BRN_CHECK_ARG(w->numel == numel, "w->numel=%lld, expected C*F=%lld", (long long)w->numel, (long long)numel);
    BRN_CHECK_ARG(w->mu && w->rho && w->dmu && w->drho, "w: NULL parameter pointer");
    BRN_CHECK_ARG(!with_prior || w->tied || (w->prior_loc && w->prior_scale), "prior_loc/prior_scale required when not tied");
    const int S = r->s_local;
    if (S == 0) return 0;
    const bool use_tc = linear_use_tc(likelihood, N, F, C, S);
    LinearWorkspace ws(workspace, numel, S, N, F, use_tc, device_sm_count());
    BRN_CHECK_ARG(workspace && workspace_bytes >= ws.bytes, "workspace too small: %zu < %zu", workspace_bytes, ws.bytes);
    set_variant(use_tc ? "tcgen05" : "simt");

    const float* eps = w->eps;
    StageTimer* st = new StageTimer("linear.sample_weights", stream);
    if (!eps) {
        if (int e = launch_philox_fill(ws.eps, numel, numel, w->var_id, *r, stream)) return e;
        eps = ws.eps;
    }
    if (int e = launch_sample_weights(w->mu, w->rho, eps, numel, ws.W, numel, numel, S, stream)) return e;
    if (!use_tc) BRN_CUDA_OK(cudaMemsetAsync(ws.dW, 0, sizeof(float) * (size_t)S * numel, stream));
    delete st;
    if (N > 0 && use_tc) {
        if (int e = launch_linear_tc(X, reinterpret_cast<const float*>(y), N, F, S, ws.W, ws.dW, -1.0f / (float)r->s_total, loss,
                                     ws.tc, "linear.split_operands", "linear.fused", stream, px))
            return e;
    } else if (N > 0) {
        StageTimer st2("linear.fused", stream);
        if (int e = launch_linear_fused(X, y, likelihood, N, F, C, S, ws.W, ws.dW, 1.0f / (float)r->s_total, loss, stream)) return e;
    } else if (use_tc) {
        BRN_CUDA_OK(cudaMemsetAsync(ws.dW, 0, sizeof(float) * (size_t)S * numel, stream));
    }
    StageTimer st3("linear.reduce_finalize", stream);
    return launch_mf_reduce_finalize(*w, eps, numel, ws.dW, numel, ws.stats, *r, with_prior, loss, stream);
}

// ---------------------------------------------------------------------------------------------
// Bayesian linear regression: y_b ~ Normal / Cauchy / Laplace(w_s . x_b, sigma_s) (see include/brancher_cuda.h,
// brn_linreg_elbo_fwd_bwd_lik).  Normal and Laplace are separable in sigma: the kernels that read X never see it, they produce
// G_s = sum_b r_sb x_b and R_s = sum_b r_sb^2 (Laplace: sum_b sign(r_sb) x_b and sum_b |r_sb|) per sample, and
// linreg_finish_kernel applies the noise scale.  Cauchy is not (d ll / d r = 2 r / (sigma^2 + r^2)): its kernels read sigma_s
// from the array linreg_sigma_kernel writes, which the finisher reads too, so the two stages cannot disagree on it.
// ---------------------------------------------------------------------------------------------
namespace brn {

// What the X pass of S weight vectors (linreg_x_pass) reads and writes besides the vectors and their gradient
struct LinregXPassBuffers {
    double* R;                 // [S] sums of squared residuals (Cauchy: of log1p(z^2); Laplace: of |r|)
    float* sigma;              // [S] noise scale per vector
    double* T;                 // [S] Cauchy: sums of z^2 / (1 + z^2)
    LinearFlashBuffers flash;
    void carve(WorkspaceCarver& take, int S, int64_t N, int F, bool flash_path, int sms) {
        R = reinterpret_cast<double*>(take(2 * (size_t)S));
        sigma = take((size_t)S);
        T = reinterpret_cast<double*>(take(2 * (size_t)S));
        flash = LinearFlashBuffers();
        if (flash_path) {
            flash.carve(take, S, F, sms);
            flash.Xh = reinterpret_cast<__half*>(take(((size_t)N * F + 1) / 2));
            flash.Xl = reinterpret_cast<__half*>(take(((size_t)N * F + 1) / 2));
        }
    }
};

struct LinregWorkspace {
    float *eps, *W, *dW, *stats;
    LinregXPassBuffers x;
    size_t bytes;
    LinregWorkspace(void* base, int S, int64_t N, int F, bool flash_path, int sms) {
        WorkspaceCarver take(base);
        eps = take((size_t)S * F);
        W = take((size_t)S * F);
        dW = take((size_t)S * F);
        stats = take(4 * (size_t)((F + 3) / 4 * 4));
        x.carve(take, S, N, F, flash_path, sms);
        bytes = take.off;
    }
};

// the one-pass kernel where the Bernoulli evaluation of the same shape takes it; there is no staged-GEMM-pair variant
static bool linreg_use_flash(const float* X, int64_t N, int F, int S) {
    return linear_use_tc(0, N, F, 1, S) && linear_flash_ok(X, N, F, S);
}

// sigma [s] = the noise scale of sample s: the constant *noise_scale, or nu_s = exp(m + softplus(rho) e_s) of the LogNormal latent
__global__ void __launch_bounds__(256)
linreg_sigma_kernel(float* __restrict__ sigma, brn_mf_var nu, int has_nu, const float* __restrict__ noise_scale, brn_sample_range r) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= r.s_local) return;
    if (has_nu) {
        const float e = nu.eps ? nu.eps[s] : philox_normal1(r.seed, philox_offset(r), nu.var_id, (uint32_t)(r.s0 + s), 0);
        sigma[s] = expf(__fmaf_rn(e, softplusf(nu.rho[0]), nu.mu[0]));
    } else {
        sigma[s] = *noise_scale;
    }
}

// The per-vector finishing formulas shared by the mean-field finisher and the particle / vector finisher, so the two families
// cannot disagree.  linreg_grad_scale: the factor that turns the X pass's G_s into d ll_s / d w_s.  linreg_loglik: ll_s from the
// X pass's sums (R_s, and T_s for Cauchy) and, in *gu, d ll_s / d u_s with u_s = log sigma_s (formulas below).
__device__ __forceinline__ float linreg_grad_scale(int lik, float sigma) {
    return lik == BRN_LINREG_CAUCHY ? 2.0f / sigma : lik == BRN_LINREG_LAPLACE ? 1.0f / sigma : 1.0f / (sigma * sigma);
}
__device__ __forceinline__ double linreg_loglik(int lik, double sd, double Rs, const double* __restrict__ T, int s, int64_t N,
                                                double* gu) {
    double ll;
    if (lik == BRN_LINREG_CAUCHY) {
        ll = -(double)N * (log(sd) + 1.1447298858494002) - Rs;                     // log pi
        *gu = 2.0 * T[s] - (double)N;
    } else if (lik == BRN_LINREG_LAPLACE) {
        const double a = Rs / sd;
        ll = -(double)N * (log(sd) + 0.6931471805599453) - a;                      // log 2
        *gu = a - (double)N;
    } else {
        const double inv_s2 = 1.0 / (sd * sd);
        ll = -0.5 * Rs * inv_s2 - (double)N * (log(sd) + (double)BRN_HALF_LOG_2PI);
        *gu = Rs * inv_s2 - (double)N;
    }
    return ll;
}

// One thread per element (s, f) of the per-sample gradient rows: dW_s *= 1 / sigma_s^2 in place (Cauchy: 2 / sigma_s, Laplace:
// 1 / sigma_s).  The thread of f == 0 also owns sample s's scalar terms, all scaled by 1 / S_total (the partial contract of
// brn_mf_normal_prior_entropy, so sharded samples sum to the unsharded result), with u_s = log sigma_s:
//   Normal   ll_s = -R_s / (2 sigma_s^2) - N u_s - N log sqrt(2 pi)   d ll_s / d u_s = R_s / sigma_s^2 - N
//   Cauchy   ll_s = -N (log pi + u_s) - R_s                            d ll_s / d u_s = 2 T_s - N
//   Laplace  ll_s = -N (log 2 + u_s) - R_s / sigma_s                   d ll_s / d u_s = R_s / sigma_s - N
// and, for the LogNormal latent (u_s = m + softplus(rho) e_s, sigma_s = exp(u_s)), d ll_s / d u_s chained to
// (m, rho), with log p(nu_s) = NORMAL_LP(log nu_s; a, b) - log nu_s and H[q(nu)] = H_Normal(softplus(rho)) + m composed as the
// scalar-DAG family composes them (tied: a = m, b = softplus(rho), differentiated through both the sample and the prior, where
// the terms cancel in closed form as in the mean-field finalisation).  lik: BRN_LINREG_NORMAL / _CAUCHY / _LAPLACE.
__global__ void __launch_bounds__(256)
linreg_finish_kernel(float* __restrict__ dW, const double* __restrict__ R, const double* __restrict__ T,
                     const float* __restrict__ sig, int lik, int F, int64_t N, brn_mf_var nu, int has_nu, brn_sample_range r,
                     int with_prior, double* __restrict__ loss) {
    __shared__ double red[32];
    __shared__ float red_m[32], red_s[32];
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t total = (int64_t)r.s_local * F;
    double elbo = 0.0;
    float gm = 0.f, gs = 0.f;            // d ELBO_s / d m, d ELBO_s / d softplus(rho) of the noise latent
    if (i < total) {
        const int s = (int)(i / F);
        const float sigma = sig[s];
        float e = 0.f, m = 0.f, sg = 1.f;
        if (has_nu) {
            e = nu.eps ? nu.eps[s] : philox_normal1(r.seed, philox_offset(r), nu.var_id, (uint32_t)(r.s0 + s), 0);
            m = nu.mu[0];
            sg = softplusf(nu.rho[0]);
        }
        dW[i] *= linreg_grad_scale(lik, sigma);
        if (i % F == 0) {
            double gu_ll;                      // d ll_s / d u_s
            elbo = linreg_loglik(lik, sigma, R[s], T, s, N, &gu_ll);
            if (has_nu) {
                const float gu = (float)gu_ll;
                gm = gu;
                gs = gu * e;
                if (with_prior) {
                    const float lx = logf(sigma);                      // LOG(EXP(u)): the sample's log as the DAG evaluates it
                    const float a = nu.tied ? m : nu.prior_loc[0], b = nu.tied ? sg : nu.prior_scale[0];
                    const float dd = lx - a, ib2 = 1.0f / (b * b);
                    const float lp = -0.5f * dd * dd * ib2 - logf(b) - BRN_HALF_LOG_2PI - lx;
                    const float ent = 0.5f + BRN_HALF_LOG_2PI + logf(sg) + m;
                    elbo += (double)lp + (double)ent;
                    if (nu.tied) {
                        // log p = -e^2/2 - log sg - c - u with a = m, b = sg: d/dm = -1, d/dsg = -1/sg - e; with the entropy's
                        // +1, +1/sg the (m, sg) gradient of prior + entropy is (0, -e) exactly
                        gs -= e;
                    } else {
                        const float gpu = -dd * ib2 - 1.0f;            // d log p / d u
                        gm += gpu + 1.0f;
                        gs += gpu * e + 1.0f / sg;
                    }
                }
            }
        }
    }
    const double tot = block_sum<double>(elbo, red);
    if (threadIdx.x == 0 && tot != 0.0) atomicAdd(loss, -tot / (double)r.s_total);
    if (has_nu) {
        const float tm = block_sum<float>(gm, red_m), ts = block_sum<float>(gs, red_s);
        if (threadIdx.x == 0) {
            const float inv_S = 1.0f / (float)r.s_total;
            atomicAdd(nu.dmu, -tm * inv_S);
            atomicAdd(nu.drho, -ts * inv_S * sigmoidf(nu.rho[0]));
        }
    }
}

// The finisher of n weight vectors (particles, or WVGD's draws) at a fixed noise scale: one thread per element (k, f) of G,
// G_k *= the likelihood's scale (G may be NULL); the thread of f == 0 computes ll_k in fp64 and writes ll[k] (ll != NULL) or adds
// -ll_k to *loss.  No 1/S factor: particle losses are sums over the particles.
__global__ void __launch_bounds__(256)
linreg_vectors_finish_kernel(float* __restrict__ G, const double* __restrict__ R, const double* __restrict__ T,
                             const float* __restrict__ sig, int lik, int F, int64_t N, int n, double* __restrict__ ll,
                             double* __restrict__ loss) {
    __shared__ double red[32];
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double nll = 0.0;
    if (i < (int64_t)n * F) {
        const int k = (int)(i / F);
        const float sigma = sig[k];
        if (G) G[i] *= linreg_grad_scale(lik, sigma);
        if (i % F == 0) {
            double gu;
            const double l = linreg_loglik(lik, sigma, R[k], T, k, N, &gu);
            if (ll) ll[k] = l;
            else nll = -l;
        }
    }
    if (loss) {
        const double tot = block_sum<double>(nll, red);
        if (threadIdx.x == 0 && tot != 0.0) atomicAdd(loss, tot);
    }
}

}  // namespace brn

// The X pass of the regression likelihood for S weight vectors W [S][F] at the noise scales b.sigma: zeroes the sums b.R (and b.T
// for Cauchy), then runs the one-pass kernel, or linear_fused_kernel on a zeroed G.  G leaves holding + d ll / d W before the
// noise scale is applied (linreg_grad_scale); with G == NULL only the sums are formed.
static int linreg_x_pass(const LinregXPassBuffers& b, int likelihood, bool use_flash, const float* X, const void* px, const float* y,
                         int64_t N, int F, const float* W, int S, float* G, cudaStream_t stream) {
    BRN_CUDA_OK(cudaMemsetAsync(b.R, 0, sizeof(double) * (size_t)S, stream));
    if (likelihood == BRN_LINREG_CAUCHY) BRN_CUDA_OK(cudaMemsetAsync(b.T, 0, sizeof(double) * (size_t)S, stream));
    if (use_flash) return launch_linear_flash(likelihood, X, px, y, N, F, S, W, G, 0.f, nullptr, b.R, b.sigma, b.T, b.flash, stream);
    if (G) BRN_CUDA_OK(cudaMemsetAsync(G, 0, sizeof(float) * (size_t)S * F, stream));      // the finishers read G even when N == 0
    if (N == 0) return 0;
    return launch_linear_fused(X, y, likelihood, N, F, 1, S, W, G, 0.f, nullptr, stream, b.R, b.sigma, b.T);
}

extern "C" size_t brn_linreg_workspace_bytes(int64_t N, int F, int s_local) {
    if (N < 0 || F <= 0 || s_local < 0) return 0;
    // sized for the one-pass kernel whenever a call of this shape may take it (X's alignment is not known here)
    return LinregWorkspace(nullptr, s_local, N, F, linreg_use_flash(nullptr, N, F, s_local), device_sm_count()).bytes;
}

extern "C" int brn_linreg_elbo_fwd_bwd(const float* X, const void* px, const float* y, int64_t N, int F, const brn_mf_var* w,
                                       const brn_mf_var* nu, const float* noise_scale, const brn_sample_range* r,
                                       void* workspace, size_t workspace_bytes, int with_prior, double* loss, void* stream_) {
    return brn_linreg_elbo_fwd_bwd_lik(X, px, y, BRN_LINREG_NORMAL, N, F, w, nu, noise_scale, r, workspace, workspace_bytes,
                                       with_prior, loss, stream_);
}

extern "C" int brn_linreg_elbo_fwd_bwd_lik(const float* X, const void* px, const float* y, int likelihood, int64_t N, int F,
                                           const brn_mf_var* w, const brn_mf_var* nu, const float* noise_scale,
                                           const brn_sample_range* r, void* workspace, size_t workspace_bytes, int with_prior,
                                           double* loss, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    BRN_CHECK_ARG(likelihood == BRN_LINREG_NORMAL || likelihood == BRN_LINREG_CAUCHY || likelihood == BRN_LINREG_LAPLACE,
                  "brn_linreg_elbo_fwd_bwd: unknown likelihood %d (Normal %d, Cauchy %d, Laplace %d)", likelihood, BRN_LINREG_NORMAL,
                  BRN_LINREG_CAUCHY, BRN_LINREG_LAPLACE);
    BRN_CHECK_ARG(w && r && loss, "brn_linreg_elbo_fwd_bwd: NULL pointer");
    BRN_CHECK_ARG(N >= 0 && F > 0, "brn_linreg_elbo_fwd_bwd: bad shape N=%lld F=%d", (long long)N, F);
    BRN_CHECK_ARG(N == 0 || (X && y), "brn_linreg_elbo_fwd_bwd: NULL data pointer");
    BRN_CHECK_ARG(F <= LN_T, "brn_linreg_elbo_fwd_bwd: F=%d exceeds the supported maximum %d", F, LN_T);
    if (int e = check_prepared_x("brn_linreg_elbo_fwd_bwd", px, N, F)) return e;
    BRN_CHECK_ARG((nu == nullptr) != (noise_scale == nullptr),
                  "brn_linreg_elbo_fwd_bwd: give exactly one of nu (LogNormal noise latent) and noise_scale (fixed noise)");
    if (int e = check_sample_range(*r)) return e;
    BRN_CHECK_ARG(w->numel == F, "w->numel=%lld, expected F=%d", (long long)w->numel, F);
    BRN_CHECK_ARG(w->mu && w->rho && w->dmu && w->drho, "w: NULL parameter pointer");
    BRN_CHECK_ARG(!with_prior || w->tied || (w->prior_loc && w->prior_scale), "w: prior_loc/prior_scale required when not tied");
    if (nu) {
        BRN_CHECK_ARG(nu->numel == 1, "nu->numel=%lld, the noise latent is a scalar", (long long)nu->numel);
        BRN_CHECK_ARG(nu->mu && nu->rho && nu->dmu && nu->drho, "nu: NULL parameter pointer");
        BRN_CHECK_ARG(!with_prior || nu->tied || (nu->prior_loc && nu->prior_scale), "nu: prior_loc/prior_scale required when not tied");
    }
    const int S = r->s_local;
    if (S == 0) return 0;
    const bool use_flash = N > 0 && linreg_use_flash(X, N, F, S);
    LinregWorkspace ws(workspace, S, N, F, use_flash, device_sm_count());
    BRN_CHECK_ARG(workspace && workspace_bytes >= ws.bytes, "workspace too small: %zu < %zu", workspace_bytes, ws.bytes);
    set_variant(use_flash ? "tcgen05-flash" : "simt");

    const float* eps = w->eps;
    {
        StageTimer st("linreg.sample_weights", stream);
        if (!eps) {
            if (int e = launch_philox_fill(ws.eps, F, F, w->var_id, *r, stream)) return e;
            eps = ws.eps;
        }
        if (int e = launch_sample_weights(w->mu, w->rho, eps, F, ws.W, F, F, S, stream)) return e;
        linreg_sigma_kernel<<<(unsigned)((S + 255) / 256), 256, 0, stream>>>(ws.x.sigma, nu ? *nu : brn_mf_var{}, nu != nullptr,
                                                                            noise_scale, *r);
        BRN_LAUNCH_OK("linreg_sigma_kernel");
    }
    {
        std::optional<StageTimer> st;       // N == 0 only zeroes the sums and dW: no X pass to time
        if (N > 0) st.emplace("linreg.fused", stream);
        if (int e = linreg_x_pass(ws.x, likelihood, use_flash, X, px, y, N, F, ws.W, S, ws.dW, stream)) return e;
    }
    {
        StageTimer st("linreg.finish", stream);
        const int64_t tot = (int64_t)S * F;
        brn_mf_var nv = nu ? *nu : brn_mf_var{};
        linreg_finish_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, stream>>>(ws.dW, ws.x.R, ws.x.T, ws.x.sigma, likelihood, F, N, nv,
                                                                              nu != nullptr, *r, with_prior, loss);
        BRN_LAUNCH_OK("linreg_finish_kernel");
    }
    StageTimer st3("linreg.reduce_finalize", stream);
    return launch_mf_reduce_finalize(*w, eps, F, ws.dW, F, ws.stats, *r, with_prior, loss, stream);
}

// ---------------------------------------------------------------------------------------------
// K4a / K6b for regression particles and vectors (brn_linreg_particles_loss_grad, brn_linreg_vectors_loglik_grad): the K2g X pass
// with the n particles as the weight vectors at a fixed noise scale, then linreg_vectors_finish_kernel instead of the mean-field
// finisher.  G (when given) leaves holding + d ll / d theta; the callers negate it and add the prior (particles_prior_kernel).
// ---------------------------------------------------------------------------------------------
static int linreg_vectors_check(const char* fn, const float* X, const void* px, const float* y, int likelihood, int64_t N, int F,
                                const float* V, int n, const float* noise_scale) {
    BRN_CHECK_ARG(likelihood == BRN_LINREG_NORMAL || likelihood == BRN_LINREG_CAUCHY || likelihood == BRN_LINREG_LAPLACE,
                  "%s: unknown likelihood %d (Normal %d, Cauchy %d, Laplace %d)", fn, likelihood, BRN_LINREG_NORMAL, BRN_LINREG_CAUCHY,
                  BRN_LINREG_LAPLACE);
    BRN_CHECK_ARG((V || n == 0) && noise_scale, "%s: NULL pointer (weight vectors or noise_scale)", fn);
    BRN_CHECK_ARG(N >= 0 && F > 0 && n >= 0, "%s: bad shape N=%lld F=%d n=%d", fn, (long long)N, F, n);
    BRN_CHECK_ARG(N == 0 || (X && y), "%s: NULL data pointer", fn);
    BRN_CHECK_ARG(F <= LN_T, "%s: F=%d exceeds the supported maximum %d", fn, F, LN_T);
    return check_prepared_x(fn, px, N, F);
}

static int linreg_vectors_run(const float* X, const void* px, const float* y, int likelihood, int64_t N, int F, const float* V, int n,
                              const float* noise_scale, float* G, double* ll, double* loss, void* workspace, size_t workspace_bytes,
                              const char* stage, cudaStream_t stream) {
    const bool use_flash = N > 0 && linreg_use_flash(X, N, F, n);
    WorkspaceCarver take(workspace);
    LinregXPassBuffers b;
    b.carve(take, n, N, F, use_flash, device_sm_count());
    BRN_CHECK_ARG(workspace && workspace_bytes >= take.off, "workspace too small: %zu < %zu", workspace_bytes, take.off);
    set_variant(use_flash ? "tcgen05-flash" : "simt");
    const int64_t tot = (int64_t)n * F;
    StageTimer st(stage, stream);
    brn_sample_range r{};
    r.s_local = n;
    r.s_total = n;
    linreg_sigma_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(b.sigma, brn_mf_var{}, 0, noise_scale, r);
    BRN_LAUNCH_OK("linreg_sigma_kernel");
    if (int e = linreg_x_pass(b, likelihood, use_flash, X, px, y, N, F, V, n, G, stream)) return e;
    linreg_vectors_finish_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, stream>>>(G, b.R, b.T, b.sigma, likelihood, F, N, n, ll, loss);
    BRN_LAUNCH_OK("linreg_vectors_finish_kernel");
    return 0;
}

extern "C" size_t brn_linreg_vectors_workspace_bytes(int64_t N, int F, int n) {
    if (N < 0 || F <= 0 || n < 0) return 0;
    // sized for the one-pass kernel whenever a call of this shape may take it (X's alignment is not known here)
    WorkspaceCarver take(nullptr);
    LinregXPassBuffers b;
    b.carve(take, n, N, F, N > 0 && linreg_use_flash(nullptr, N, F, n), device_sm_count());
    return take.off;
}

extern "C" int brn_linreg_particles_loss_grad(const float* X, const void* px, const float* y, int likelihood, int64_t N, int F,
                                              const float* theta, int n, const float* prior_loc, const float* prior_scale,
                                              const float* noise_scale, float* G, double* loss, void* workspace,
                                              size_t workspace_bytes, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (int e = linreg_vectors_check("brn_linreg_particles_loss_grad", X, px, y, likelihood, N, F, theta, n, noise_scale)) return e;
    BRN_CHECK_ARG((G || n == 0) && loss, "brn_linreg_particles_loss_grad: NULL pointer (G or loss)");
    BRN_CHECK_ARG((prior_loc == nullptr) == (prior_scale == nullptr), "prior_loc and prior_scale must both be given or both NULL");
    if (n == 0) return 0;
    if (int e = linreg_vectors_run(X, px, y, likelihood, N, F, theta, n, noise_scale, G, nullptr, loss, workspace, workspace_bytes,
                                   "linreg_particles.loglik_grad", stream))
        return e;
    const int64_t total = (int64_t)n * F;
    StageTimer st("linreg_particles.prior", stream);
    particles_prior_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(theta, prior_loc, prior_scale, F, total, G, loss);
    BRN_LAUNCH_OK("particles_prior_kernel");
    return 0;
}

extern "C" int brn_linreg_vectors_loglik_grad(const float* X, const void* px, const float* y, int likelihood, int64_t N, int F,
                                              const float* V, int n, const float* noise_scale, float* G, double* ll, void* workspace,
                                              size_t workspace_bytes, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (int e = linreg_vectors_check("brn_linreg_vectors_loglik_grad", X, px, y, likelihood, N, F, V, n, noise_scale)) return e;
    BRN_CHECK_ARG(ll || n == 0, "brn_linreg_vectors_loglik_grad: NULL pointer (ll)");
    if (n == 0) return 0;
    if (int e = linreg_vectors_run(X, px, y, likelihood, N, F, V, n, noise_scale, G, ll, nullptr, workspace, workspace_bytes,
                                   "linreg_vectors.loglik_grad", stream))
        return e;
    if (G) {       // + d ll / d V -> the ABI's loss gradient - d ll / d V
        const int64_t total = (int64_t)n * F;
        particles_prior_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(V, nullptr, nullptr, F, total, G, nullptr);
        BRN_LAUNCH_OK("particles_prior_kernel");
    }
    return 0;
}
