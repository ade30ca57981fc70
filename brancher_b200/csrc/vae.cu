// K5 -- amortised VAE (include/brancher_cuda.h: brn_vae_elbo_fwd_bwd), examples/VAE_playground.py:30-80.
//
// The weights are shared by all MC samples, so every layer is an ordinary [rows x features] contraction over
// rows = s_local * B (decoder) or B (encoder).  All of them run on the tcgen05 3xTF32 GEMM of umma_gemm.cuh:
//   forward   act_i   = relu(act_{i-1} . W_i^T + b_i)                  A = act_{i-1} [rows][n_in],  B = W_i   [n_out][n_in]
//   data grad dpre_{i-1} = (dpre_i . W_i) * relu'(act_{i-1})           A = dpre_i    [rows][n_out], B = W_i^T [n_in][n_out]
//   weight grad dW_i  = dpre_i^T . act_{i-1}                            A = dpre_i    [rows][n_out], B = act_{i-1} [rows][n_in]
// with the bias / ReLU / Bernoulli likelihood / ReLU mask / bias-gradient column sums fused into the GEMM epilogues,
// which write each activation (gradient) tensor once, row-major, as one plain fp32 matrix: the forward and data-gradient
// GEMMs read it K-major and the weight-gradient GEMM MN-major, and both split it into TF32 (hi, lo) on the fly.
// The K = L (latent, 2 in the example) layers -- encoder heads, sampling, first decoder layer -- are SIMT kernels.
// Gradients are carried in "ELBO-sum units" (d sum_{s,b} elbo_sb / d .) in a zeroed scratch buffer and scaled by
// -1/(S_total*B_total) into the caller's buffers by one final launch.
#include "common.cuh"
#include "umma_gemm.cuh"

#include <math.h>
#include <stdlib.h>
#include <algorithm>

namespace brn {

constexpr int VAE_BK = 16;          // K chunk (64-byte swizzle, 5-stage TMA ring)
constexpr int VAE_MAX_L = 16;       // latent sizes supported by the SIMT kernels
constexpr int VAE_MAX_H0 = 1024;    // width of the first decoder layer supported by vae_dec0_bwd_kernel

// [rows][n] tensor as the GEMMs consume it
struct VaeAct {
    float *rm_hi, *rm_lo;     // [rows][ld]   K-major operand (K = n) of the next layer, MN-major operand (K = rows) of the weight gradient
    int64_t ld;
    int n;
};

// lane l returns sum over the warp's 32 lanes of v[l]  (31 shuffles instead of 32 x 5)
__device__ __forceinline__ float warp_colsum32(const float (&v)[32]) {
    const int lane = threadIdx.x & 31;
    float a[16], b[8], c[4], d[2];
    {
        const bool up = (lane & 16) != 0;
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            const float send = up ? v[k] : v[k + 16], keep = up ? v[k + 16] : v[k];
            a[k] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
        }
    }
    {
        const bool up = (lane & 8) != 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const float send = up ? a[k] : a[k + 8], keep = up ? a[k + 8] : a[k];
            b[k] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
        }
    }
    {
        const bool up = (lane & 4) != 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float send = up ? b[k] : b[k + 4], keep = up ? b[k + 4] : b[k];
            c[k] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
        }
    }
    {
        const bool up = (lane & 2) != 0;
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const float send = up ? c[k] : c[k + 2], keep = up ? c[k + 2] : c[k];
            d[k] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
        }
    }
    const bool up = (lane & 1) != 0;
    const float send = up ? d[0] : d[1], keep = up ? d[1] : d[0];
    return keep + __shfl_xor_sync(0xffffffffu, send, 1);
}

// write 4 consecutive columns of one row, row-major (vectorised when whole and aligned), TF32-split
// A NULL lo pointer means "this copy is ONE plain fp32 matrix" (the consuming GEMM splits it on the fly, SPLIT mask of
// umma_gemm.cuh): row-major copies are always plain here.
__device__ __forceinline__ void store_split4(const float (&v)[4], int nvalid, float* rh, float* rl) {
    float h[4], l[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) umma::split_tf32(v[j], h[j], l[j]);
    if (!rl) {
        if (nvalid >= 4) *reinterpret_cast<float4*>(rh) = make_float4(v[0], v[1], v[2], v[3]);
        else {
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (j < nvalid) rh[j] = v[j];
        }
    } else if (nvalid >= 4) {
        *reinterpret_cast<float4*>(rh) = make_float4(h[0], h[1], h[2], h[3]);
        *reinterpret_cast<float4*>(rl) = make_float4(l[0], l[1], l[2], l[3]);
    } else {
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (j < nvalid) { rh[j] = h[j]; rl[j] = l[j]; }
    }
}

// ------------------------------------------------------------------------------------------------
// epilogue: hidden layer forward.  out = relu(D + bias), row-major.
// ------------------------------------------------------------------------------------------------
struct EpiDense {
    struct Params {
        const float* bias; float *rm_hi, *rm_lo; int64_t ld; int rows, cols;
    };
    template <int CPT>
    static __device__ __forceinline__ void finish(const Params& p, float (&r)[CPT], int row, int blk, bool, int) {
        const int c0 = blk * CPT;
        if (row >= p.rows || c0 >= p.cols) return;
        const int valid = min(CPT, p.cols - c0);
        float* rh = p.rm_hi + (int64_t)row * p.ld + c0;
        float* rl = p.rm_lo ? p.rm_lo + (int64_t)row * p.ld + c0 : nullptr;
#pragma unroll
        for (int i = 0; i < CPT; i += 4) {
            if (i < valid) {
                float v[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) v[j] = (i + j < valid) ? fmaxf(r[i + j] + __ldg(p.bias + c0 + i + j), 0.f) : 0.f;
                store_split4(v, valid - i, rh + i, rl ? rl + i : nullptr);
            }
        }
    }
};

// ------------------------------------------------------------------------------------------------
// epilogue: decoder output layer + Binomial(1, logits) likelihood (distributions.py:561-575 with total_count = 1:
// the three lgamma terms vanish):   l = D + bias ;  ll += x l - (max(l,0) + log(1 + e^-|l|)) ;  d = x - sigmoid(l)
// d is written row-major; its column sums are the output bias gradient.
// ------------------------------------------------------------------------------------------------
struct EpiBern {
    struct Params {
        const float* bias; const float* X; int64_t ldx; int B;
        float *rm_hi, *rm_lo; int64_t ld; int rows, cols; double* ll; float* dbias;
    };
    template <int CPT>
    static __device__ __forceinline__ void finish(const Params& p, float (&r)[CPT], int row, int blk, bool, int) {
        const int c0 = blk * CPT;
        if (c0 >= p.cols) return;                       // warp-uniform
        const bool row_ok = row < p.rows;
        const int valid = row_ok ? min(CPT, p.cols - c0) : 0;
        const int lane = threadIdx.x & 31;
        // each thread walks its own row of X: 32 sectors per warp load, but every 128-byte line then serves the thread's next
        // 31 elements from L1.  (Measured: reading the transposed copy instead -- coalesced, no reuse -- is 38 % SLOWER.)
        const float* x = p.X + (int64_t)(row_ok ? row % p.B : 0) * p.ldx + c0;
        float* rh = p.rm_hi + (int64_t)row * p.ld + c0;
        float* rl = p.rm_lo ? p.rm_lo + (int64_t)row * p.ld + c0 : nullptr;
        float ll = 0.f;
        if (valid == CPT && (reinterpret_cast<uintptr_t>(x) & 15) == 0) {
            // full, aligned block (the common case).  The epilogue warps were stalled on the per-element x loads 57 % of the
            // time (profiles/r1o_*): here the thread's row segment is fetched as float4, FOUR groups (16 elements) ahead of use.
            constexpr int NG = CPT / 4;
            const float4* x4 = reinterpret_cast<const float4*>(x);
            float4 xn[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) xn[q] = q < NG ? __ldg(x4 + q) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int i0 = 0; i0 < CPT; i0 += 32) {
                float d32[32];
#pragma unroll
                for (int hb = 0; hb < 32; hb += 16) {
                    const int g0 = (i0 + hb) / 4;
                    float4 xc[4];
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        xc[q] = xn[q];
                        if (g0 + 4 + q < NG) xn[q] = __ldg(x4 + g0 + 4 + q);
                    }
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int i = i0 + hb + 4 * q;
                        float v[4] = {0.f, 0.f, 0.f, 0.f};
                        if (i < CPT) {
                            const float xv4[4] = {xc[q].x, xc[q].y, xc[q].z, xc[q].w};
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const float l = r[i + j] + __ldg(p.bias + c0 + i + j);
                                const float xv = xv4[j];
                                float e, inv, lg;
                                asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-1.4426950408889634f * fabsf(l)));
                                const float ope = 1.f + e;
                                asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(inv) : "f"(ope));
                                asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(ope));
                                const float sig = l >= 0.f ? inv : e * inv;
                                ll += __fmaf_rn(xv, l, -__fmaf_rn(lg, 0.6931471805599453f, fmaxf(l, 0.f)));
                                v[j] = xv - sig;
                            }
                            store_split4(v, 4, rh + i, rl ? rl + i : nullptr);
                        }
#pragma unroll
                        for (int j = 0; j < 4; ++j) d32[hb + 4 * q + j] = v[j];
                    }
                }
                const float cs = warp_colsum32(d32);
                if (c0 + i0 + lane < p.cols && i0 + lane < CPT) atomicAdd(p.dbias + c0 + i0 + lane, cs);
            }
        } else
#pragma unroll
        for (int i0 = 0; i0 < CPT; i0 += 32) {
            float d32[32];
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
                float v[4] = {0.f, 0.f, 0.f, 0.f};
                if (i0 + i < CPT && i0 + i < valid) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        if (i0 + i + j < valid) {
                            const float l = r[i0 + i + j] + __ldg(p.bias + c0 + i0 + i + j);
                            const float xv = __ldg(x + i0 + i + j);
                            float e, inv, lg;                       // MUFU ex2 / rcp / lg2: absolute errors ~1e-7
                            asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-1.4426950408889634f * fabsf(l)));
                            const float ope = 1.f + e;
                            asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(inv) : "f"(ope));
                            asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(ope));
                            const float sig = l >= 0.f ? inv : e * inv;
                            ll += __fmaf_rn(xv, l, -__fmaf_rn(lg, 0.6931471805599453f, fmaxf(l, 0.f)));
                            v[j] = xv - sig;
                        }
                    }
                    store_split4(v, valid - i0 - i, rh + i0 + i, rl ? rl + i0 + i : nullptr);
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) d32[i + j] = v[j];
            }
            const float cs = warp_colsum32(d32);
            if (c0 + i0 + lane < p.cols && i0 + lane < CPT) atomicAdd(p.dbias + c0 + i0 + lane, cs);
        }
        double tot = (double)ll;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, o);
        if (lane == 0 && tot != 0.0) atomicAdd(p.ll, tot);
    }
};

// ------------------------------------------------------------------------------------------------
// epilogue: data gradient.  g = D * [mask > 0]  (mask = the hi part of the layer's ReLU output), written row-major
// (to `plain` when it is set: the first decoder layer's SIMT backward reads that);
// column sums of g = the layer's bias gradient.
// ------------------------------------------------------------------------------------------------
struct EpiMask {
    struct Params {
        const float* mask; int64_t ldm; float *rm_hi, *rm_lo; int64_t ld; float* plain; int64_t ldp;
        int rows, cols; float* dbias;
    };
    template <int CPT>
    static __device__ __forceinline__ void finish(const Params& p, float (&r)[CPT], int row, int blk, bool, int) {
        const int c0 = blk * CPT;
        if (c0 >= p.cols) return;                       // warp-uniform
        const bool row_ok = row < p.rows;
        const int valid = row_ok ? min(CPT, p.cols - c0) : 0;
        const int lane = threadIdx.x & 31;
        const float* mk = p.mask + (int64_t)(row_ok ? row : 0) * p.ldm + c0;
        // full, aligned block (the common case): the thread's row segment of the mask is fetched as float4, FOUR groups (16
        // elements) ahead of use -- with per-element loads on demand the data-gradient GEMMs ran at 17-26 % tensor activity
        // (profiles/r2f_ncu_full_vae_summary.txt), as EpiBern did before the same change
        const bool fast = valid == CPT && (reinterpret_cast<uintptr_t>(mk) & 15) == 0;
        constexpr int NG = CPT / 4;
        const float4* m4 = reinterpret_cast<const float4*>(mk);
        float4 mn[4];
        if (fast) {
#pragma unroll
            for (int q = 0; q < 4; ++q) mn[q] = q < NG ? __ldg(m4 + q) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int i0 = 0; i0 < CPT; i0 += 32) {
            float d32[32];
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
                float v[4] = {0.f, 0.f, 0.f, 0.f};
                if (i0 + i < CPT && i0 + i < valid) {
                    if (fast) {
                        const int gq = (i0 + i) / 4;                // compile-time: the loops are fully unrolled
                        const float4 mc = mn[gq & 3];
                        if (gq + 4 < NG) mn[gq & 3] = __ldg(m4 + gq + 4);
                        v[0] = mc.x > 0.f ? r[i0 + i] : 0.f;
                        v[1] = mc.y > 0.f ? r[i0 + i + 1] : 0.f;
                        v[2] = mc.z > 0.f ? r[i0 + i + 2] : 0.f;
                        v[3] = mc.w > 0.f ? r[i0 + i + 3] : 0.f;
                    } else {
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        if (i0 + i + j < valid) v[j] = __ldg(mk + i0 + i + j) > 0.f ? r[i0 + i + j] : 0.f;
                    }
                    const int col = i0 + i;
                    if (p.plain) {
                        float* o = p.plain + (int64_t)row * p.ldp + c0 + col;
                        if (valid - col >= 4) *reinterpret_cast<float4*>(o) = make_float4(v[0], v[1], v[2], v[3]);
                        else {
#pragma unroll
                            for (int j = 0; j < 4; ++j)
                                if (col + j < valid) o[j] = v[j];
                        }
                    } else {
                        store_split4(v, valid - col, p.rm_hi + (int64_t)row * p.ld + c0 + col,
                                     p.rm_lo ? p.rm_lo + (int64_t)row * p.ld + c0 + col : nullptr);
                    }
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) d32[i + j] = v[j];
            }
            const float cs = warp_colsum32(d32);
            if (c0 + i0 + lane < p.cols && i0 + lane < CPT) atomicAdd(p.dbias + c0 + i0 + lane, cs);
        }
    }
};

// N tile: 128 with SIXTEEN epilogue warps when N is a multiple of 128 (every hidden width of C5: the epilogues -- bias / ReLU /
// mask / split stores -- are the bound of these GEMMs, and twice the warps at half the columns per thread hide their latency);
// otherwise the narrowest instantiated width that covers N in ceil(N / 208) tiles, eight epilogue warps.
static int pick_bn(int N) {
    if (N % 128 == 0) return -128;
    const int nt = (N + 207) / 208, per = (N + nt - 1) / nt;
    return per <= 128 ? 128 : (per <= 176 ? 176 : 208);
}

template <class Epi>
static int launch_gemm(const float* Ah, const float* Al, int M, int64_t lda, const float* Bh, const float* Bl, int N, int64_t ldb,
                       int K, int mode, const typename Epi::Params& ep, cudaStream_t stream, bool allow_split = false) {
    switch (pick_bn(N)) {
        // every A operand of K5 (activations, gradients) is one plain fp32 matrix: SPLIT = 1, two converter warps (they split
        // the plain fp32 A tile into the TF32 pair inside the stage)
        case -128: return launch_umma_nt<128, VAE_BK, Epi, 16, 1, 2>(Ah, nullptr, M, lda, Bh, Bl, N, ldb, K, mode, 2, ep, stream, allow_split);
        case 128: return launch_umma_nt<128, VAE_BK, Epi, UG_EPI_WARPS, 1, 2>(Ah, nullptr, M, lda, Bh, Bl, N, ldb, K, mode, 2, ep, stream,
                                                                           allow_split);
        case 176: return launch_umma_nt<176, VAE_BK, Epi, UG_EPI_WARPS, 1, 2>(Ah, nullptr, M, lda, Bh, Bl, N, ldb, K, mode, 2, ep, stream,
                                                                           allow_split);
        default: return launch_umma_nt<208, VAE_BK, Epi, UG_EPI_WARPS, 1, 2>(Ah, nullptr, M, lda, Bh, Bl, N, ldb, K, mode, 2, ep, stream,
                                                                          allow_split);
    }
}

// ------------------------------------------------------------------------------------------------
// SIMT kernels for the K = L layers
// ------------------------------------------------------------------------------------------------
// encoder heads (VAE_playground.py:44-46): mean = W_mean h + b_mean ; sd = softplus(W_sd h + b_sd) + sd_offset ; analytic
// entropy of Qz summed over latent dims (variables.py:156-162), counted once per (sample, row).  One warp per row.
__global__ void vae_heads_fwd_kernel(const float* __restrict__ a_hi, const float* __restrict__ a_lo, int64_t ld, int B, int h, int L,
                                     const float* __restrict__ Wm, const float* __restrict__ bm, const float* __restrict__ Ws,
                                     const float* __restrict__ bs, float sd_offset, float* __restrict__ mean, float* __restrict__ sd,
                                     float* __restrict__ sdpre, double* ent_acc, float s_local) {
    const int row = (int)((blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (row >= B) return;
    float ent = 0.f;
    for (int l = 0; l < L; ++l) {
        float pm = 0.f, ps = 0.f;
        for (int j = lane; j < h; j += 32) {
            const float a = a_hi[(int64_t)row * ld + j] + (a_lo ? a_lo[(int64_t)row * ld + j] : 0.f);
            pm = __fmaf_rn(a, Wm[(int64_t)l * h + j], pm);
            ps = __fmaf_rn(a, Ws[(int64_t)l * h + j], ps);
        }
        pm = warp_sum(pm); ps = warp_sum(ps);
        if (lane == 0) {
            const float m = pm + bm[l], sp = ps + bs[l], s = softplusf(sp) + sd_offset;
            mean[(int64_t)row * L + l] = m; sd[(int64_t)row * L + l] = s; sdpre[(int64_t)row * L + l] = sp;
            ent += 0.5f + BRN_HALF_LOG_2PI + logf(s);
        }
    }
    if (lane == 0) atomicAdd(ent_acc, (double)ent * (double)s_local);
}

__device__ __forceinline__ float dec0_value(const float* zs, const float* __restrict__ V0, const float* __restrict__ c0, int L, int j) {
    float v = c0[j];
    for (int l = 0; l < L; ++l) v = __fmaf_rn(zs[l], V0[(int64_t)j * L + l], v);
    return fmaxf(v, 0.f);
}

// z = mean + eps * sd (Normal.rsample, distributions.py:122), log p(z) = sum_lat N(z; 0, 1), and the first decoder layer
// g_0 = relu(V_0 z + c_0) written row-major as plain fp32.  32 rows (row = s * B + b) per block.
__global__ void __launch_bounds__(256)
vae_sample_dec0_kernel(const float* __restrict__ mean, const float* __restrict__ sd, const float* __restrict__ eps_in, int B, int L,
                       int R, int64_t row0_global, brn_sample_range r, uint32_t var_id, const float* __restrict__ V0,
                       const float* __restrict__ c0, int h0, float* __restrict__ z, float* __restrict__ epsb, VaeAct a0,
                       double* lpz_acc) {
    extern __shared__ float zs[];          // [32][L]
    __shared__ float red[32];
    const int r0 = blockIdx.x * 32, tid = threadIdx.x;
    float lp = 0.f;
    for (int idx = tid; idx < 32 * L; idx += 256) {
        const int row = r0 + idx / L, l = idx % L;
        float zz = 0.f;
        if (row < R) {
            const int s = row / B, b = row % B;
            const float e = eps_in ? eps_in[(int64_t)row * L + l]
                                   : philox_normal1(r.seed, philox_offset(r), var_id, (uint32_t)(r.s0 + s), (row0_global + b) * L + l);
            zz = __fmaf_rn(e, sd[(int64_t)b * L + l], mean[(int64_t)b * L + l]);
            z[(int64_t)row * L + l] = zz;
            epsb[(int64_t)row * L + l] = e;
            lp += -0.5f * zz * zz - BRN_HALF_LOG_2PI;
        }
        zs[idx] = zz;
    }
    __syncthreads();
    const float tot = block_sum(lp, red);
    if (tid == 0 && tot != 0.f) atomicAdd(lpz_acc, (double)tot);
    for (int idx = tid; idx < 32 * h0; idx += 256) {            // consecutive threads -> consecutive columns
        const int rr = idx / h0, j = idx % h0, row = r0 + rr;
        if (row < R) {
            a0.rm_hi[(int64_t)row * a0.ld + j] = dec0_value(zs + rr * L, V0, c0, L, j);
        }
    }
}

// backward of the first decoder layer and of the sampling step.  dpre0 [R][ld0] (already ReLU-masked):
//   gV0[j][l] += sum_r dpre0[r][j] z[r][l] ;  dz[r][l] = sum_j dpre0[r][j] V0[j][l] - z[r][l]   (the -z is d log N(z;0,1)/dz)
//   dmean[b][l] += dz ;  dsd[b][l] += dz * eps                                            (z = mean + sd * eps)
constexpr int DEC0_RC = 64;
template <int LP, int JPT>
__global__ void __launch_bounds__(256)
vae_dec0_bwd_kernel(const float* __restrict__ dpre0, int64_t ld0, const float* __restrict__ z, const float* __restrict__ epsb,
                    const float* __restrict__ V0, int h0, int L, int R, int B, float* gV0, float* dmean, float* dsd) {
    __shared__ float zs[DEC0_RC][LP], dzs[DEC0_RC][LP];
    const int r0 = blockIdx.x * DEC0_RC, tid = threadIdx.x, lane = tid & 31;
    for (int idx = tid; idx < DEC0_RC * LP; idx += 256) {
        const int rr = idx / LP, l = idx % LP, row = r0 + rr;
        zs[rr][l] = (row < R && l < L) ? z[(int64_t)row * L + l] : 0.f;
        dzs[rr][l] = 0.f;
    }
    float vreg[JPT][LP], acc[JPT][LP];
#pragma unroll
    for (int jj = 0; jj < JPT; ++jj) {
        const int j = tid + 256 * jj;
#pragma unroll
        for (int l = 0; l < LP; ++l) {
            vreg[jj][l] = (j < h0 && l < L) ? V0[(int64_t)j * L + l] : 0.f;
            acc[jj][l] = 0.f;
        }
    }
    __syncthreads();
    const int nrows = min(DEC0_RC, R - r0);
    for (int rr = 0; rr < nrows; ++rr) {
        const float* g = dpre0 + (int64_t)(r0 + rr) * ld0;
        float part[LP];
#pragma unroll
        for (int l = 0; l < LP; ++l) part[l] = 0.f;
#pragma unroll
        for (int jj = 0; jj < JPT; ++jj) {
            const int j = tid + 256 * jj;
            const float gv = j < h0 ? g[j] : 0.f;
#pragma unroll
            for (int l = 0; l < LP; ++l) {
                acc[jj][l] = __fmaf_rn(gv, zs[rr][l], acc[jj][l]);
                part[l] = __fmaf_rn(gv, vreg[jj][l], part[l]);
            }
        }
#pragma unroll
        for (int l = 0; l < LP; ++l) {
            if (l < L) {
                const float p = warp_sum(part[l]);
                if (lane == 0) atomicAdd(&dzs[rr][l], p);
            }
        }
    }
    __syncthreads();
#pragma unroll
    for (int jj = 0; jj < JPT; ++jj) {
        const int j = tid + 256 * jj;
        if (j < h0) {
#pragma unroll
            for (int l = 0; l < LP; ++l)
                if (l < L) atomicAdd(gV0 + (int64_t)j * L + l, acc[jj][l]);
        }
    }
    for (int idx = tid; idx < nrows * L; idx += 256) {
        const int rr = idx / L, l = idx % L, row = r0 + rr, b = row % B;
        const float dzv = dzs[rr][l] - zs[rr][l];
        atomicAdd(dmean + (int64_t)b * L + l, dzv);
        atomicAdd(dsd + (int64_t)b * L + l, dzv * epsb[(int64_t)row * L + l]);
    }
}

// backward of the encoder heads: entropy gradient, softplus chain rule, head weight / bias gradients, and the gradient
// w.r.t. the last hidden layer's pre-activation (ReLU-masked, row-major plain fp32) + that layer's bias gradient.
template <int LP>
__global__ void __launch_bounds__(256)
vae_heads_bwd_kernel(const float* __restrict__ dmean, const float* __restrict__ dsd, const float* __restrict__ sd,
                     const float* __restrict__ sdpre, int B, int L, float s_local, const float* __restrict__ a_hi,
                     const float* __restrict__ a_lo, int64_t lda, const float* __restrict__ Wm, const float* __restrict__ Ws, int h,
                     VaeAct dpre, float* gWm, float* gWs, float* gbm, float* gbs, float* gb_last) {
    __shared__ float dm[32][LP], dsp[32][LP];
    const int b0 = blockIdx.x * 32, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    for (int idx = tid; idx < 32 * LP; idx += 256) {
        const int rr = idx / LP, l = idx % LP, b = b0 + rr;
        float m = 0.f, sp = 0.f;
        if (b < B && l < L) {
            const int64_t o = (int64_t)b * L + l;
            m = dmean[o];
            sp = (dsd[o] + s_local / sd[o]) * sigmoidf(sdpre[o]);      // d softplus(x)/dx = sigmoid(x)
        }
        dm[rr][l] = m; dsp[rr][l] = sp;
    }
    __syncthreads();
    if (tid < 2 * L) {
        const int l = tid % L;
        float s = 0.f;
        for (int rr = 0; rr < 32; ++rr) s += tid < L ? dm[rr][l] : dsp[rr][l];
        atomicAdd((tid < L ? gbm : gbs) + l, s);
    }
    for (int c0 = w * 32; c0 < h; c0 += 8 * 32) {
        const int j = c0 + lane;
        const bool jok = j < h;
        float wm[LP], wsd[LP], am[LP], as[LP];
#pragma unroll
        for (int l = 0; l < LP; ++l) {
            wm[l] = (jok && l < L) ? Wm[(int64_t)l * h + j] : 0.f;
            wsd[l] = (jok && l < L) ? Ws[(int64_t)l * h + j] : 0.f;
            am[l] = 0.f; as[l] = 0.f;
        }
        float colsum = 0.f;
        for (int rr = 0; rr < 32; ++rr) {
            const int b = b0 + rr;
            if (jok && b < B) {
                const float ahi = a_hi[(int64_t)b * lda + j], a = ahi + (a_lo ? a_lo[(int64_t)b * lda + j] : 0.f);
                float g = 0.f;
#pragma unroll
                for (int l = 0; l < LP; ++l) {
                    g = __fmaf_rn(dm[rr][l], wm[l], g);
                    g = __fmaf_rn(dsp[rr][l], wsd[l], g);
                    am[l] = __fmaf_rn(dm[rr][l], a, am[l]);
                    as[l] = __fmaf_rn(dsp[rr][l], a, as[l]);
                }
                const float v = ahi > 0.f ? g : 0.f;
                dpre.rm_hi[(int64_t)b * dpre.ld + j] = v;
                colsum += v;
            }
        }
        if (jok) {
            atomicAdd(gb_last + j, colsum);
#pragma unroll
            for (int l = 0; l < LP; ++l) {
                if (l < L) {
                    atomicAdd(gWm + (int64_t)l * h + j, am[l]);
                    atomicAdd(gWs + (int64_t)l * h + j, as[l]);
                }
            }
        }
    }
}

// caller's gradient buffers += scale * scratch gradients; loss += scale * (ll + log p(z) + entropy) + constant
struct VaeGradTable {
    int n;
    float* dst[40];
    int64_t off[40], numel[40];
};
__global__ void vae_finalize_kernel(const __grid_constant__ VaeGradTable t, const float* __restrict__ tmp, float scale,
                                    const double* __restrict__ acc, double* loss, double add_const) {
    const int k = blockIdx.y;
    float* dst = t.dst[k];
    const float* src = tmp + t.off[k];
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < t.numel[k]; i += (int64_t)gridDim.x * blockDim.x)
        dst[i] += scale * src[i];
    if (blockIdx.x == 0 && k == 0 && threadIdx.x == 0) *loss += (double)scale * (acc[0] + acc[1] + acc[2]) + add_const;
}

// ------------------------------------------------------------------------------------------------
// workspace
// ------------------------------------------------------------------------------------------------
struct VaeWeights {          // TF32-split weight matrix [n_out][n_in] in both K-major layouts + its scratch gradients
    float *hi, *lo, *t_hi, *t_lo;
    int64_t ld, ldt;
    float *gW, *gb;
    int64_t offW, offb;
};

static inline int64_t pad4l(int64_t n) { return (n + 3) / 4 * 4; }

struct VaeWorkspace {
    VaeAct Xa, enc_a[BRN_VAE_MAX_HIDDEN], enc_d[BRN_VAE_MAX_HIDDEN], dec_a[BRN_VAE_MAX_HIDDEN], dec_d[BRN_VAE_MAX_HIDDEN], dL;
    VaeWeights encW[BRN_VAE_MAX_HIDDEN], decW[BRN_VAE_MAX_HIDDEN], outW, meanW, sdW;
    float *dpre0; int64_t ld0;
    float *mean, *sd, *sdpre, *z, *epsb;
    // zeroed region
    char* zero_begin; size_t zero_bytes;
    float *dmean, *dsd, *grads; int64_t grads_numel;
    double* acc;
    size_t bytes;

    VaeWorkspace(void* base, const brn_vae_model& m, int B, int S) {
        WorkspaceCarver take(base);
        // ONE plain fp32 matrix (rm_lo == NULL): the GEMMs that read it split it on the fly (SPLIT mask of umma_gemm.cuh)
        auto act = [&](VaeAct& a, int64_t rows, int n) {
            a.n = n; a.ld = pad4l(n);
            a.rm_hi = take((size_t)rows * a.ld); a.rm_lo = nullptr;
        };
        const int64_t R = (int64_t)S * B;
        act(Xa, B, m.D);
        for (int i = 0; i < m.n_enc; ++i) { act(enc_a[i], B, m.enc[i].n_out); act(enc_d[i], B, m.enc[i].n_out); }
        for (int i = 0; i < m.n_dec; ++i) {
            act(dec_a[i], R, m.dec[i].n_out);
            if (i > 0) act(dec_d[i], R, m.dec[i].n_out);
        }
        act(dL, R, m.D);
        ld0 = pad4l(m.dec[0].n_out);
        dpre0 = take((size_t)R * ld0);
        mean = take((size_t)B * m.L); sd = take((size_t)B * m.L); sdpre = take((size_t)B * m.L);
        z = take((size_t)R * m.L); epsb = take((size_t)R * m.L);
        auto wsplit = [&](VaeWeights& w, const brn_dense_layer& l, bool gemm) {
            w.ld = pad4l(l.n_in); w.ldt = pad4l(l.n_out);
            w.hi = w.lo = w.t_hi = w.t_lo = nullptr;
            if (gemm) {
                w.hi = take((size_t)l.n_out * w.ld); w.lo = take((size_t)l.n_out * w.ld);
                w.t_hi = take((size_t)l.n_in * w.ldt); w.t_lo = take((size_t)l.n_in * w.ldt);
            }
        };
        for (int i = 0; i < m.n_enc; ++i) wsplit(encW[i], m.enc[i], true);
        for (int i = 0; i < m.n_dec; ++i) wsplit(decW[i], m.dec[i], i > 0);
        wsplit(outW, m.dec_out, true);
        wsplit(meanW, m.enc_mean, false);
        wsplit(sdW, m.enc_sd, false);
        // zeroed region: scratch gradients (flat), dmean/dsd, scalar accumulators
        const size_t zb = take.off;
        int64_t g = 0;
        auto gslot = [&](VaeWeights& w, const brn_dense_layer& l) {
            w.offW = g; g += pad4l((int64_t)l.n_out * l.n_in);
            w.offb = g; g += pad4l(l.n_out);
        };
        for (int i = 0; i < m.n_enc; ++i) gslot(encW[i], m.enc[i]);
        gslot(meanW, m.enc_mean); gslot(sdW, m.enc_sd);
        for (int i = 0; i < m.n_dec; ++i) gslot(decW[i], m.dec[i]);
        gslot(outW, m.dec_out);
        grads_numel = g;
        grads = take((size_t)g);
        dmean = take((size_t)B * m.L); dsd = take((size_t)B * m.L);
        acc = reinterpret_cast<double*>(take.bytes(4 * sizeof(double)));
        zero_begin = base ? reinterpret_cast<char*>(base) + zb : nullptr;
        zero_bytes = take.off - zb;
        auto gptr = [&](VaeWeights& w) { w.gW = grads ? grads + w.offW : nullptr; w.gb = grads ? grads + w.offb : nullptr; };
        for (int i = 0; i < m.n_enc; ++i) gptr(encW[i]);
        for (int i = 0; i < m.n_dec; ++i) gptr(decW[i]);
        gptr(outW); gptr(meanW); gptr(sdW);
        bytes = take.off;
    }
};

static int check_layer(const brn_dense_layer& l, int n_in, int n_out, const char* what, int i) {
    BRN_CHECK_ARG(l.W && l.b && l.dW && l.db, "brn_vae: %s[%d]: NULL pointer", what, i);
    BRN_CHECK_ARG(l.n_in == n_in && l.n_out == n_out && n_out > 0, "brn_vae: %s[%d] is %d -> %d, expected %d -> %d", what, i, l.n_in,
                  l.n_out, n_in, n_out);
    return 0;
}

static int validate(const brn_vae_model* m) {
    BRN_CHECK_ARG(m, "brn_vae: NULL model");
    BRN_CHECK_ARG(m->D > 0 && m->L > 0 && m->L <= VAE_MAX_L, "brn_vae: D=%d L=%d (latent size must be 1..%d)", m->D, m->L, VAE_MAX_L);
    BRN_CHECK_ARG(m->n_enc >= 1 && m->n_enc <= BRN_VAE_MAX_HIDDEN && m->n_dec >= 1 && m->n_dec <= BRN_VAE_MAX_HIDDEN,
                  "brn_vae: n_enc=%d n_dec=%d (1..%d hidden layers each)", m->n_enc, m->n_dec, BRN_VAE_MAX_HIDDEN);
    int n = m->D;
    for (int i = 0; i < m->n_enc; ++i) { if (int e = check_layer(m->enc[i], n, m->enc[i].n_out, "enc", i)) return e; n = m->enc[i].n_out; }
    if (int e = check_layer(m->enc_mean, n, m->L, "enc_mean", 0)) return e;
    if (int e = check_layer(m->enc_sd, n, m->L, "enc_sd", 0)) return e;
    n = m->L;
    for (int i = 0; i < m->n_dec; ++i) { if (int e = check_layer(m->dec[i], n, m->dec[i].n_out, "dec", i)) return e; n = m->dec[i].n_out; }
    if (int e = check_layer(m->dec_out, n, m->D, "dec_out", 0)) return e;
    BRN_CHECK_ARG(m->dec[0].n_out <= VAE_MAX_H0, "brn_vae: first decoder layer wider than %d", VAE_MAX_H0);
    return 0;
}

template <int LP>
static int launch_dec0_bwd(int h0, const float* dpre0, int64_t ld0, const float* z, const float* epsb, const float* V0, int L, int64_t R,
                           int B, float* gV0, float* dmean, float* dsd, cudaStream_t stream) {
    const unsigned grid = (unsigned)((R + DEC0_RC - 1) / DEC0_RC);
    if (h0 <= 512) vae_dec0_bwd_kernel<LP, 2><<<grid, 256, 0, stream>>>(dpre0, ld0, z, epsb, V0, h0, L, (int)R, B, gV0, dmean, dsd);
    else vae_dec0_bwd_kernel<LP, 4><<<grid, 256, 0, stream>>>(dpre0, ld0, z, epsb, V0, h0, L, (int)R, B, gV0, dmean, dsd);
    BRN_LAUNCH_OK("vae_dec0_bwd_kernel");
    return 0;
}

}  // namespace brn

using namespace brn;

extern "C" size_t brn_vae_workspace_bytes(const brn_vae_model* m, int B, int s_local) {
    if (!m || B <= 0 || s_local < 0 || validate(m) != 0) return 0;
    return VaeWorkspace(nullptr, *m, B, s_local).bytes;
}

extern "C" int brn_vae_elbo_fwd_bwd(const float* X, int B, int64_t row0, int64_t B_total, const brn_vae_model* m, const float* eps,
                                    uint32_t var_id, const brn_sample_range* r, void* workspace, size_t workspace_bytes,
                                    int add_constant, double* loss, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    BRN_CHECK_ARG(X && m && r && loss, "brn_vae_elbo_fwd_bwd: NULL pointer");
    if (int e = validate(m)) return e;
    BRN_CHECK_ARG(B > 0 && row0 >= 0 && row0 + B <= B_total, "brn_vae_elbo_fwd_bwd: bad row range row0=%lld B=%d B_total=%lld",
                  (long long)row0, B, (long long)B_total);
    if (int e = check_sample_range(*r)) return e;
    const int S = r->s_local, L = m->L, D = m->D;
    if (S == 0) return 0;
    const int64_t R = (int64_t)S * B;
    BRN_CHECK_ARG(R < (1ll << 31), "brn_vae_elbo_fwd_bwd: s_local * B = %lld rows exceed 2^31", (long long)R);
    VaeWorkspace ws(workspace, *m, B, S);
    BRN_CHECK_ARG(workspace && workspace_bytes >= ws.bytes, "workspace too small: %zu < %zu", workspace_bytes, ws.bytes);
    set_variant("tcgen05");
    BRN_CUDA_OK(cudaMemsetAsync(ws.zero_begin, 0, ws.zero_bytes, stream));
    double* acc_ll = ws.acc, *acc_lpz = ws.acc + 1, *acc_ent = ws.acc + 2;

    // 0. operands: X as a plain row-major copy, every weight matrix a GEMM reads TF32-split in both K-major layouts
    {
        StageTimer st("vae.split_operands", stream);
        BRN_CUDA_OK(cudaMemcpy2DAsync(ws.Xa.rm_hi, ws.Xa.ld * sizeof(float), X, D * sizeof(float), D * sizeof(float), B,
                                      cudaMemcpyDeviceToDevice, stream));         // plain row-major copy with the padded pitch
        auto wsplit = [&](const brn_dense_layer& l, VaeWeights& w) {
            return launch_split_tf32(l.W, l.n_in, l.n_out, l.n_in, w.hi, w.lo, w.ld, w.t_hi, w.t_lo, w.ldt, stream);
        };
        for (int i = 0; i < m->n_enc; ++i) if (int e = wsplit(m->enc[i], ws.encW[i])) return e;
        for (int i = 1; i < m->n_dec; ++i) if (int e = wsplit(m->dec[i], ws.decW[i])) return e;
        if (int e = wsplit(m->dec_out, ws.outW)) return e;
    }
    auto dense_fwd = [&](const VaeAct& in, int64_t rows, const brn_dense_layer& l, const VaeWeights& w, VaeAct& out) {
        EpiDense::Params ep;
        ep.bias = l.b; ep.rm_hi = out.rm_hi; ep.rm_lo = out.rm_lo; ep.ld = out.ld;
        ep.rows = (int)rows; ep.cols = l.n_out;
        return launch_gemm<EpiDense>(in.rm_hi, in.rm_lo, (int)rows, in.ld, w.hi, w.lo, l.n_out, w.ld, l.n_in, 2, ep, stream);
    };
    // dpre_prev = (dpre . W) * relu'(a_prev)  [+ bias gradient of the previous layer]
    auto data_grad = [&](const VaeAct& dcur, int64_t rows, const brn_dense_layer& l, const VaeWeights& w, const VaeAct& a_prev,
                         VaeAct* dprev, float* plain, int64_t ldp, float* gb_prev) {
        EpiMask::Params ep;
        ep.mask = a_prev.rm_hi; ep.ldm = a_prev.ld;
        ep.rm_hi = dprev ? dprev->rm_hi : nullptr; ep.rm_lo = dprev ? dprev->rm_lo : nullptr;
        ep.ld = dprev ? dprev->ld : 0; ep.plain = plain; ep.ldp = ldp;
        ep.rows = (int)rows; ep.cols = l.n_in; ep.dbias = gb_prev;
        return launch_gemm<EpiMask>(dcur.rm_hi, dcur.rm_lo, (int)rows, dcur.ld, w.t_hi, w.t_lo, l.n_in, w.ldt, l.n_out, 2, ep, stream);
    };
    // gW = dpre^T . a_in, read MN-major from the row-major tensors (launch_umma_tn_plain: no transposed copies)
    // (K = rows: few output tiles, so the K range is split over the SMs with atomic partial sums)
    auto weight_grad = [&](const VaeAct& dcur, const VaeAct& a_in, int64_t rows, const brn_dense_layer& l, float* gW) {
        EpiStore::Params ep;
        constexpr int cpt = 64;        // columns per epilogue thread of both variants below
        ep.out = gW; ep.rows = l.n_out; ep.row_stride = l.n_in; ep.col_stride = 1; ep.blk_stride = cpt; ep.blk_valid = cpt;
        ep.col_limit = l.n_in; ep.total_blks = (l.n_in + cpt - 1) / cpt;
        // N tile 256 with sixteen epilogue and eight converter warps where the layer's input width allows it (measured at C5:
        // 1.745 ms per evaluation against 1.78 with 128-column tiles)
        if (l.n_in % 256 == 0)
            return launch_umma_tn_plain<256, VAE_BK, EpiStore, 16, 8>(dcur.rm_hi, l.n_out, dcur.ld, a_in.rm_hi, l.n_in, a_in.ld,
                                                                      (int)rows, 0, 2, ep, stream, true);
        return launch_umma_tn_plain<128, VAE_BK, EpiStore, UG_EPI_WARPS, 4>(dcur.rm_hi, l.n_out, dcur.ld, a_in.rm_hi, l.n_in, a_in.ld,
                                                                            (int)rows, 0, 2, ep, stream, true);
    };

    // 1. encoder forward
    {
        StageTimer st("vae.encoder_fwd", stream);
        const VaeAct* in = &ws.Xa;
        for (int i = 0; i < m->n_enc; ++i) {
            if (int e = dense_fwd(*in, B, m->enc[i], ws.encW[i], ws.enc_a[i])) return e;
            in = &ws.enc_a[i];
        }
        const int h = m->enc[m->n_enc - 1].n_out;
        vae_heads_fwd_kernel<<<(B + 7) / 8, 256, 0, stream>>>(in->rm_hi, in->rm_lo, in->ld, B, h, L, m->enc_mean.W, m->enc_mean.b,
                                                             m->enc_sd.W, m->enc_sd.b, m->sd_offset, ws.mean, ws.sd, ws.sdpre, acc_ent,
                                                             (float)S);
        BRN_LAUNCH_OK("vae_heads_fwd_kernel");
    }
    // 2. sample z, log p(z), first decoder layer
    {
        StageTimer st("vae.sample_dec0", stream);
        const unsigned grid = (unsigned)((R + 31) / 32);
        vae_sample_dec0_kernel<<<grid, 256, 32 * L * sizeof(float), stream>>>(ws.mean, ws.sd, eps, B, L, (int)R, row0, *r, var_id,
                                                                              m->dec[0].W, m->dec[0].b, m->dec[0].n_out, ws.z, ws.epsb,
                                                                              ws.dec_a[0], acc_lpz);
        BRN_LAUNCH_OK("vae_sample_dec0_kernel");
    }
    // 3. decoder forward + likelihood
    {
        StageTimer st("vae.decoder_fwd", stream);
        for (int i = 1; i < m->n_dec; ++i)
            if (int e = dense_fwd(ws.dec_a[i - 1], R, m->dec[i], ws.decW[i], ws.dec_a[i])) return e;
        const VaeAct& in = ws.dec_a[m->n_dec - 1];
        EpiBern::Params ep;
        ep.bias = m->dec_out.b; ep.X = X; ep.ldx = D; ep.B = B;
        ep.rm_hi = ws.dL.rm_hi; ep.rm_lo = ws.dL.rm_lo; ep.ld = ws.dL.ld;
        ep.rows = (int)R; ep.cols = D; ep.ll = acc_ll; ep.dbias = ws.outW.gb;
        if (int e = launch_gemm<EpiBern>(in.rm_hi, in.rm_lo, (int)R, in.ld, ws.outW.hi, ws.outW.lo, D, ws.outW.ld, m->dec_out.n_in, 2, ep,
                                         stream))
            return e;
    }
    // 4. decoder backward
    {
        StageTimer st("vae.decoder_bwd", stream);
        const VaeAct* dcur = &ws.dL;
        for (int i = m->n_dec; i >= 1; --i) {              // layer i: dec[i] for i < n_dec, the output layer for i == n_dec
            const brn_dense_layer& l = i == m->n_dec ? m->dec_out : m->dec[i];
            VaeWeights& w = i == m->n_dec ? ws.outW : ws.decW[i];
            const VaeAct& a_prev = ws.dec_a[i - 1];
            if (int e = weight_grad(*dcur, a_prev, R, l, w.gW)) return e;
            if (i - 1 == 0) {
                if (int e = data_grad(*dcur, R, l, w, a_prev, nullptr, ws.dpre0, ws.ld0, ws.decW[0].gb)) return e;
            } else {
                if (int e = data_grad(*dcur, R, l, w, a_prev, &ws.dec_d[i - 1], nullptr, 0, ws.decW[i - 1].gb)) return e;
                dcur = &ws.dec_d[i - 1];
            }
        }
    }
    // 5. first decoder layer + sampling backward
    {
        StageTimer st("vae.dec0_bwd", stream);
        const int h0 = m->dec[0].n_out;
        int e = 0;
        if (L <= 2) e = launch_dec0_bwd<2>(h0, ws.dpre0, ws.ld0, ws.z, ws.epsb, m->dec[0].W, L, R, B, ws.decW[0].gW, ws.dmean, ws.dsd, stream);
        else if (L <= 4) e = launch_dec0_bwd<4>(h0, ws.dpre0, ws.ld0, ws.z, ws.epsb, m->dec[0].W, L, R, B, ws.decW[0].gW, ws.dmean, ws.dsd, stream);
        else if (L <= 8) e = launch_dec0_bwd<8>(h0, ws.dpre0, ws.ld0, ws.z, ws.epsb, m->dec[0].W, L, R, B, ws.decW[0].gW, ws.dmean, ws.dsd, stream);
        else e = launch_dec0_bwd<16>(h0, ws.dpre0, ws.ld0, ws.z, ws.epsb, m->dec[0].W, L, R, B, ws.decW[0].gW, ws.dmean, ws.dsd, stream);
        if (e) return e;
    }
    // 6. encoder backward
    {
        StageTimer st("vae.encoder_bwd", stream);
        const int last = m->n_enc - 1, h = m->enc[last].n_out;
        const VaeAct& a = ws.enc_a[last];
        const unsigned grid = (unsigned)((B + 31) / 32);
#define BRN_HEADS_BWD(LP)                                                                                                            \
    vae_heads_bwd_kernel<LP><<<grid, 256, 0, stream>>>(ws.dmean, ws.dsd, ws.sd, ws.sdpre, B, L, (float)S, a.rm_hi, a.rm_lo, a.ld,     \
                                                       m->enc_mean.W, m->enc_sd.W, h, ws.enc_d[last], ws.meanW.gW, ws.sdW.gW,       \
                                                       ws.meanW.gb, ws.sdW.gb, ws.encW[last].gb)
        if (L <= 2) BRN_HEADS_BWD(2);
        else if (L <= 4) BRN_HEADS_BWD(4);
        else if (L <= 8) BRN_HEADS_BWD(8);
        else BRN_HEADS_BWD(16);
#undef BRN_HEADS_BWD
        BRN_LAUNCH_OK("vae_heads_bwd_kernel");
        for (int i = last; i >= 0; --i) {
            const VaeAct& a_in = i == 0 ? ws.Xa : ws.enc_a[i - 1];
            if (int e = weight_grad(ws.enc_d[i], a_in, B, m->enc[i], ws.encW[i].gW)) return e;
            if (i > 0)
                if (int e = data_grad(ws.enc_d[i], B, m->enc[i], ws.encW[i], ws.enc_a[i - 1], &ws.enc_d[i - 1], nullptr, 0, ws.encW[i - 1].gb))
                    return e;
        }
    }
    // 7. scale into the caller's gradient buffers, finish the loss
    {
        StageTimer st("vae.finalize", stream);
        VaeGradTable t;
        t.n = 0;
        int64_t maxn = 1;
        auto add = [&](const brn_dense_layer& l, const VaeWeights& w) {
            t.dst[t.n] = l.dW; t.off[t.n] = w.offW; t.numel[t.n] = (int64_t)l.n_out * l.n_in; ++t.n;
            t.dst[t.n] = l.db; t.off[t.n] = w.offb; t.numel[t.n] = l.n_out; ++t.n;
            maxn = std::max(maxn, (int64_t)l.n_out * l.n_in);
        };
        for (int i = 0; i < m->n_enc; ++i) add(m->enc[i], ws.encW[i]);
        add(m->enc_mean, ws.meanW); add(m->enc_sd, ws.sdW);
        for (int i = 0; i < m->n_dec; ++i) add(m->dec[i], ws.decW[i]);
        add(m->dec_out, ws.outW);
        const float scale = (float)(-1.0 / ((double)r->s_total * (double)B_total));
        const double cst = add_constant ? -log((double)r->s_total) : 0.0;
        dim3 grid((unsigned)std::min<int64_t>((maxn + 255) / 256, 64), t.n);
        vae_finalize_kernel<<<grid, 256, 0, stream>>>(t, ws.grads, scale, ws.acc, loss, cst);
        BRN_LAUNCH_OK("vae_finalize_kernel");
    }
    return 0;
}
