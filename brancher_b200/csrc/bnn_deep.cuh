// K3 with 2..4 hidden layers: brn_bnn_deep_*.  Included by bnn.cu after the two-layer code, whose layer-1 stages and head
// it reuses:
//   1. sampling of all 2L+2 variables (W1 through the layer-1 sampler of its variant, the rest in groups of <= 4)
//   2. layer-1 GEMM                   pre_1 = X W1_s^T, SIMT or tcgen05 by the two-layer rule on H1
//   3. forward stages l = 2..L        h_{l-1} = act(pre_{l-1} + b_{l-1}),  pre_l = h_{l-1} W_l,s^T          (bnn_deep_fwd_kernel)
//   4. head                           bnn_mid2_kernel<false> on a layout view: logits, log-softmax, loss, dW_out, db_out,
//                                     db_L and dpre_L
//   5. backward stages l = L..2       dh_{l-1} = dpre_l W_l,s,  dpre_{l-1} = dh_{l-1} act'(h_{l-1}),
//                                     dW_l,s += dpre_l^T h_{l-1},  db_{l-1} += sum_rows dpre_{l-1}           (bnn_deep_bwd_kernel)
//   6. layer-1 weight-gradient GEMM   dW1_s = dpre_1^T X
//   7. sample-axis reduction, prior, entropy and chain rule, in groups of <= 4 consecutive variables
// Stages 3 and 5 run on the warp-level tensor cores (mma.sync m16n8k8 TF32, 3-product hi/lo split as bnn_mid4_kernel):
// one CTA = 128 batch rows of one sample, 16 warps; the sample's W_l sits in shared memory.
#pragma once

namespace brn {

constexpr int DEEP_MAXL = 4, DEEP_MAXH = 128, DEEP_R = 128, DEEP_THREADS = 512;
constexpr int SC_DPRE = 4;            // scal slot: max |dpre_1| of the tcgen05 layer-1 variant's weight-gradient GEMM

// per-sample row of the sampled weights / noise / gradients: W1, b1, W2, b2, ..., W_L, b_L, W_out, b_out, each variable at a
// 16-byte aligned offset (so the grouped statistics launches take their vector path)
struct DeepLayout {
    int B, P, C, L;
    int H[DEEP_MAXL], act[DEEP_MAXL];
    int64_t off[2 * DEEP_MAXL + 2], n[2 * DEEP_MAXL + 2];
    int64_t numel, ldw;
    int nvars() const { return 2 * L + 2; }
    DeepLayout(int B_, int P_, int L_, const int* H_, const int* act_, int C_) : B(B_), P(P_), C(C_), L(L_) {
        int64_t o = 0;
        for (int l = 0; l <= L; ++l) {
            const int rows = l < L ? H_[l] : C, cols = l == 0 ? P : H_[l - 1];
            if (l < L) { H[l] = H_[l]; act[l] = act_ ? act_[l] : 0; }
            n[2 * l] = (int64_t)rows * cols;
            n[2 * l + 1] = rows;
            off[2 * l] = o;
            o += (n[2 * l] + 3) / 4 * 4;
            off[2 * l + 1] = o;
            o += (n[2 * l + 1] + 3) / 4 * 4;
        }
        numel = off[2 * L + 1] + n[2 * L + 1];
        ldw = o;
    }
    // the head's view: the two-layer layout over (b_L, W_out, b_out) of this row
    BnnLayout head() const {
        BnnLayout V(B, P, H[L - 1], C, act[L - 1]);
        V.ob1 = off[2 * L - 1]; V.oW2 = off[2 * L]; V.ob2 = off[2 * L + 1];
        V.numel = numel; V.ldw = ldw;
        return V;
    }
};

__host__ __device__ __forceinline__ int pad8(int x) { return (x + 7) & ~7; }
__host__ __device__ __forceinline__ int pad16(int x) { return (x + 15) & ~15; }

// shared-memory pitches are 4 mod 8 words: the fragment loads (8 rows g x 4 columns t) hit 32 distinct banks
static size_t deep_fwd_smem(int Hin, int Hout) {
    return sizeof(float) * ((size_t)DEEP_R * (pad8(Hin) + 4) + (size_t)pad8(Hout) * (pad8(Hin) + 4));
}
static size_t deep_bwd_smem(int Hin, int Hout) {
    const size_t pd = pad16(Hout) + 4, ph = pad8(Hin) + 4;
    return sizeof(float) * ((size_t)DEEP_R * pd + (size_t)DEEP_R * ph + (size_t)pad8(Hin) * pd + 8 * (size_t)pad8(Hin));
}

__device__ __forceinline__ void split3(float x, float& hi, float& lo) { split_tf32_trunc_lo(x, hi, lo); }

// ---------------------------------------------------------------------------------------------------
// forward stage: h = act(pre_in + b) for this CTA's 128 rows (kept in shared memory, stored for the backward stage), then
// pre_out[b, n] = sum_k h[b, k] W[n, k].  Warp w: rows 16 (w & 7) .. +16, output n-tiles (w >> 3) + 2 jj.
// PRE_T: pre_in is [S][Hin][B] (tcgen05 layer-1 output), else [S][B][Hin].
// ---------------------------------------------------------------------------------------------------
template <bool PRE_T>
__global__ void __launch_bounds__(DEEP_THREADS, 1)
bnn_deep_fwd_kernel(const float* __restrict__ pre_in, const float* __restrict__ Wall, int64_t ldw, int64_t oW, int64_t ob, int B,
                    int Hin, int Hout, int act, float* __restrict__ h_out, float* __restrict__ pre_out) {
    extern __shared__ __align__(16) float sm[];
    const int KP = pad8(Hin), NP = pad8(Hout), ph = KP + 4;
    float* hs = sm;                                  // [128][ph]
    float* ws = hs + (size_t)DEEP_R * ph;            // [NP][ph]
    const int s = blockIdx.y, b0 = blockIdx.x * DEEP_R, tid = threadIdx.x;
    const float* Ws = Wall + (int64_t)s * ldw;
    for (int idx = tid; idx < NP * KP; idx += DEEP_THREADS) {
        const int nn = idx / KP, k = idx - nn * KP;
        ws[nn * ph + k] = (nn < Hout && k < Hin) ? Ws[oW + (int64_t)nn * Hin + k] : 0.f;
    }
    const float* ps = pre_in + (int64_t)s * B * Hin;
    for (int idx = tid; idx < DEEP_R * KP; idx += DEEP_THREADS) {
        int r, k;
        if (PRE_T) { k = idx / DEEP_R; r = idx - k * DEEP_R; }
        else { r = idx / KP; k = idx - r * KP; }
        float v = 0.f;
        if (b0 + r < B && k < Hin)
            v = act_exact(act, (PRE_T ? ps[(int64_t)k * B + b0 + r] : ps[(int64_t)(b0 + r) * Hin + k]) + Ws[ob + k]);
        hs[r * ph + k] = v;
    }
    __syncthreads();
    float* hs_out = h_out + ((int64_t)s * B + b0) * Hin;
    for (int idx = tid; idx < DEEP_R * Hin; idx += DEEP_THREADS) {
        const int r = idx / Hin, k = idx - r * Hin;
        if (b0 + r < B) hs_out[idx] = hs[r * ph + k];
    }

    const int warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    const int rg = warp & 7, nh = warp >> 3, NT = NP / 8;
    float hh[8][4], cr[8][4];
#pragma unroll
    for (int j = 0; j < 8; ++j)
#pragma unroll
        for (int i = 0; i < 4; ++i) hh[j][i] = cr[j][i] = 0.f;
    const float* arow = hs + (16 * rg + g) * ph + t;
    const float* brow = ws + g * ph + t;
    for (int kk = 0; kk < KP / 8; ++kk) {
        float ahi[4], alo[4];
        split3(arow[8 * kk], ahi[0], alo[0]);
        split3(arow[8 * kk + 8 * ph], ahi[1], alo[1]);
        split3(arow[8 * kk + 4], ahi[2], alo[2]);
        split3(arow[8 * kk + 8 * ph + 4], ahi[3], alo[3]);
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) {
            const int j = nh + 2 * jj;
            if (j < NT) {
                float bh0, bl0, bh1, bl1;
                split3(brow[8 * j * ph + 8 * kk], bh0, bl0);
                split3(brow[8 * j * ph + 8 * kk + 4], bh1, bl1);
                mma_tf32(hh[jj], ahi, bh0, bh1);
                mma_tf32(cr[jj], alo, bh0, bh1);
                mma_tf32(cr[jj], ahi, bl0, bl1);
            }
        }
    }
    const int r0 = b0 + 16 * rg + g, r1 = r0 + 8;
    float* po = pre_out + (int64_t)s * B * Hout;
#pragma unroll
    for (int jj = 0; jj < 8; ++jj) {
        const int c = 8 * (nh + 2 * jj) + 2 * t;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int rr = i < 2 ? r0 : r1, cc = c + (i & 1);
            if (rr < B && cc < Hout) po[(int64_t)rr * Hout + cc] = hh[jj][i] + cr[jj][i];
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// backward stage of layer l (W [Hout][Hin] = W_l, h = h_{l-1}), one CTA = 128 rows of one sample:
//   (a) dh[b, i] = sum_j dpre[b, j] W[j, i];  dpre_out[b, i] = dh act'(h[b, i]);  db[i] += sum_b dpre_out[b, i]
//   (b) dW[j, i] += sum_b dpre[b, j] h[b, i]
// dpre_out may alias nothing the CTA reads.  ABSMAX: max |dpre_out| into *amax (the tcgen05 weight-gradient GEMM's bound).
// ---------------------------------------------------------------------------------------------------
template <bool ABSMAX>
__global__ void __launch_bounds__(DEEP_THREADS, 1)
bnn_deep_bwd_kernel(const float* __restrict__ dpre, const float* __restrict__ h, const float* __restrict__ Wall, float* __restrict__ dWall,
                    int64_t ldw, int64_t oW, int64_t ob, int B, int Hin, int Hout, int act, float* __restrict__ dpre_out,
                    float* __restrict__ amax) {
    extern __shared__ __align__(16) float sm[];
    const int KO = pad16(Hout), KP = pad8(Hin), pd = KO + 4, ph = KP + 4;
    float* ds = sm;                                  // [128][pd]   dpre, columns >= Hout zero
    float* hs = ds + (size_t)DEEP_R * pd;            // [128][ph]   h, rows >= B and columns >= Hin zero
    float* wt = hs + (size_t)DEEP_R * ph;            // [KP][pd]    W^T
    float* cs = wt + (size_t)KP * pd;                // [8][KP]     per-row-group column sums of dpre_out
    const int s = blockIdx.y, b0 = blockIdx.x * DEEP_R, tid = threadIdx.x;
    const float* Ws = Wall + (int64_t)s * ldw;
    float* dWs = dWall + (int64_t)s * ldw;
    for (int idx = tid; idx < KO * KP; idx += DEEP_THREADS) {        // coalesced along i
        const int j = idx / KP, i = idx - j * KP;
        wt[i * pd + j] = (j < Hout && i < Hin) ? Ws[oW + (int64_t)j * Hin + i] : 0.f;
    }
    const float* dps = dpre + ((int64_t)s * B + b0) * Hout;
    for (int idx = tid; idx < DEEP_R * KO; idx += DEEP_THREADS) {
        const int r = idx / KO, j = idx - r * KO;
        ds[r * pd + j] = (b0 + r < B && j < Hout) ? dps[(int64_t)r * Hout + j] : 0.f;
    }
    const float* hsrc = h + ((int64_t)s * B + b0) * Hin;
    for (int idx = tid; idx < DEEP_R * KP; idx += DEEP_THREADS) {
        const int r = idx / KP, i = idx - r * KP;
        hs[r * ph + i] = (b0 + r < B && i < Hin) ? hsrc[(int64_t)r * Hin + i] : 0.f;
    }
    __syncthreads();

    const int warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    const int rg = warp & 7, nh = warp >> 3, NT = KP / 8;
    float m = 0.f;
    {   // (a)
        float hh[8][4], cr[8][4];
#pragma unroll
        for (int j = 0; j < 8; ++j)
#pragma unroll
            for (int i = 0; i < 4; ++i) hh[j][i] = cr[j][i] = 0.f;
        const float* arow = ds + (16 * rg + g) * pd + t;
        const float* brow = wt + g * pd + t;
        for (int kk = 0; kk < KO / 8; ++kk) {
            float ahi[4], alo[4];
            split3(arow[8 * kk], ahi[0], alo[0]);
            split3(arow[8 * kk + 8 * pd], ahi[1], alo[1]);
            split3(arow[8 * kk + 4], ahi[2], alo[2]);
            split3(arow[8 * kk + 8 * pd + 4], ahi[3], alo[3]);
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) {
                const int j = nh + 2 * jj;
                if (j < NT) {
                    float bh0, bl0, bh1, bl1;
                    split3(brow[8 * j * pd + 8 * kk], bh0, bl0);
                    split3(brow[8 * j * pd + 8 * kk + 4], bh1, bl1);
                    mma_tf32(hh[jj], ahi, bh0, bh1);
                    mma_tf32(cr[jj], alo, bh0, bh1);
                    mma_tf32(cr[jj], ahi, bl0, bl1);
                }
            }
        }
        const int rl0 = 16 * rg + g, rl1 = rl0 + 8;
        float* po = dpre_out + ((int64_t)s * B + b0) * Hin;
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) {
            const int j = nh + 2 * jj;
            if (j < NT) {
                const int c = 8 * j + 2 * t;
                float dp[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int rl = i < 2 ? rl0 : rl1, cc = c + (i & 1);
                    dp[i] = (hh[jj][i] + cr[jj][i]) * act_grad_from_h(act, hs[rl * ph + cc]);    // 0 on pad rows / columns
                    if (b0 + rl < B && cc < Hin) po[(int64_t)rl * Hin + cc] = dp[i];
                    if (ABSMAX) m = fmaxf(m, fabsf(dp[i]));
                }
                float c0 = dp[0] + dp[2], c1 = dp[1] + dp[3];     // column sums over this warp's 16 rows
#pragma unroll
                for (int o = 4; o < 32; o <<= 1) {
                    c0 += __shfl_xor_sync(0xffffffffu, c0, o);
                    c1 += __shfl_xor_sync(0xffffffffu, c1, o);
                }
                if (g == 0) { cs[rg * KP + c] = c0; cs[rg * KP + c + 1] = c1; }
            }
        }
    }
    {   // (b): warp w owns the 16-row m-tile (w & 7) of dW and the n-tiles (w >> 3) + 2 jj
        const int mt = rg, MT = KO / 16;
        if (mt < MT) {
            float hh[8][4], cr[8][4];
#pragma unroll
            for (int j = 0; j < 8; ++j)
#pragma unroll
                for (int i = 0; i < 4; ++i) hh[j][i] = cr[j][i] = 0.f;
            const float* acol = ds + t * pd + 16 * mt + g;
            const float* bcol = hs + t * ph + g;
#pragma unroll 2
            for (int kk = 0; kk < DEEP_R / 8; ++kk) {
                float ahi[4], alo[4];
                split3(acol[8 * kk * pd], ahi[0], alo[0]);
                split3(acol[8 * kk * pd + 8], ahi[1], alo[1]);
                split3(acol[(8 * kk + 4) * pd], ahi[2], alo[2]);
                split3(acol[(8 * kk + 4) * pd + 8], ahi[3], alo[3]);
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) {
                    const int j = nh + 2 * jj;
                    if (j < NT) {
                        float bh0, bl0, bh1, bl1;
                        split3(bcol[8 * kk * ph + 8 * j], bh0, bl0);
                        split3(bcol[(8 * kk + 4) * ph + 8 * j], bh1, bl1);
                        mma_tf32(hh[jj], ahi, bh0, bh1);
                        mma_tf32(cr[jj], alo, bh0, bh1);
                        mma_tf32(cr[jj], ahi, bl0, bl1);
                    }
                }
            }
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) {
                const int c = 8 * (nh + 2 * jj) + 2 * t;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int row = 16 * mt + g + (i < 2 ? 0 : 8), col = c + (i & 1);
                    if (row < Hout && col < Hin) atomicAdd(&dWs[oW + (int64_t)row * Hin + col], hh[jj][i] + cr[jj][i]);
                }
            }
        }
    }
    __syncthreads();
    for (int i = tid; i < Hin; i += DEEP_THREADS) {
        float acc = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) acc += cs[w * KP + i];
        atomicAdd(&dWs[ob + i], acc);
    }
    if (ABSMAX) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        if (lane == 0 && m > 0.f) atomic_absmax(amax, m);
    }
}

// dpre_1 [S][B][H] fp32 -> the tcgen05 weight-gradient GEMM's K-major fp16 pairs [(s * Hp + h)][ldB], scaled by
// p2_scale(*amax); rows h in [H, Hp) zero
__global__ void bnn_deep_split_dpre_kernel(const float* __restrict__ dpre, int B, int H, int Hp, __half* __restrict__ hi,
                                           __half* __restrict__ lo, int64_t ldB, const float* __restrict__ amax) {
    __shared__ float tile[32][33];
    const float sc = p2_scale(*amax);
    const int b0 = blockIdx.x * 32, h0 = blockIdx.y * 32, s = blockIdx.z, tx = threadIdx.x, ty = threadIdx.y;   // 32 x 8
    const float* src = dpre + (int64_t)s * B * H;
    for (int i = ty; i < 32; i += 8) {
        const int b = b0 + i, hh = h0 + tx;
        tile[i][tx] = (b < B && hh < H) ? src[(int64_t)b * H + hh] : 0.f;
    }
    __syncthreads();
    for (int i = ty; i < 32; i += 8) {
        const int hh = h0 + i, b = b0 + tx;
        if (hh < Hp && b < B) {
            __half vh, vl;
            split_f16(tile[tx][i] * sc, vh, vl);
            const int64_t o = ((int64_t)s * Hp + hh) * ldB + b;
            hi[o] = vh;
            lo[o] = vl;
        }
    }
}

struct DeepWorkspace {
    float *eps, *W, *dW, *stats;
    float* pre[DEEP_MAXL];    // pre_l [S][B][H_l] (pre_1 [S][H1][B] in the tcgen05 variant), overwritten by dpre_l
    float* h[DEEP_MAXL];      // h_l [S][B][H_l], l < L
    BnnTcWorkspace tc;
    size_t bytes;
    DeepWorkspace(void* base, const DeepLayout& D, int S) {
        WorkspaceCarver take(base);
        eps = take((size_t)S * D.ldw);
        W = take((size_t)S * D.ldw);
        dW = take((size_t)S * D.ldw);
        stats = take(4 * (size_t)D.ldw);
        for (int l = 0; l < D.L; ++l) {
            pre[l] = take((size_t)S * D.B * D.H[l]);
            h[l] = l + 1 < D.L ? take((size_t)S * D.B * D.H[l]) : nullptr;
        }
        tc.carve(take, BnnLayout(D.B, D.P, D.H[0], D.C), S);
        bytes = take.off;
    }
};

static bool deep_use_tc(int H1) {
    bool use_tc = (H1 > BNN_UMMA_HP - 16 && H1 <= BNN_UMMA_HP);
    if (const char* v = getenv("BRN_BNN_VARIANT")) {
        if (!strcmp(v, "simt")) use_tc = false;
        else if (!strcmp(v, "tcgen05") && H1 <= BNN_UMMA_HP) use_tc = true;
    }
    return use_tc;
}

template <class K>
static int deep_smem_attr(K kernel, size_t smem) {
    BRN_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    return 0;
}

// stages 1 - 3 (sampling, layer-1 GEMM, forward stages): on return ws.pre[L-1] holds pre_L [S][B][H_L]
static int deep_forward(const float* X, const DeepLayout& D, const brn_mf_var* vars, const brn_sample_range* r, const DeepWorkspace& ws,
                        bool use_tc, bool zero_grads, cudaStream_t stream) {
    const int B = D.B, P = D.P, S = r->s_local, nv = D.nvars();
    {
        StageTimer st("bnn.sample_weights", stream);
        if (use_tc) {
            if (int e = bnn_tc_sample_w1(vars[0], vars[2], D.H[0], P, D.ldw, r, ws.tc, ws.eps, stream)) return e;
        } else if (int e = launch_sample_multi(vars, D.off, 1, ws.eps, ws.W, D.ldw, *r, stream)) {
            return e;
        }
        // the other variables in groups of <= 4 consecutive ones, their per-sample gradient slots zeroed (accumulated into)
        for (int v0 = 1; v0 < nv; v0 += 4)
            if (int e = launch_sample_multi(vars + v0, D.off + v0, std::min(4, nv - v0), ws.eps, ws.W, D.ldw, *r, stream,
                                            zero_grads ? ws.dW : nullptr))
                return e;
        if (use_tc) {
            if (int e = bnn_tc_split_x(X, B, P, ws.tc, stream)) return e;
        } else if (int e = wait_data_ready(stream)) {
            return e;
        }
    }
    {
        StageTimer st("bnn.gemm_fwd", stream);
        const int H1 = D.H[0];
        if (use_tc) {
            if (int e = bnn_tc_gemm_fwd(B, P, H1, S, ws.tc, ws.pre[0], stream)) return e;
        } else if (int e = launch_sgemm_batched<true, true>(X, P, 0, ws.W, P, D.ldw, ws.pre[0], H1, (int64_t)B * H1, B, H1, P, S, stream)) {
            return e;
        }
    }
    StageTimer st("bnn.deep_fwd", stream);
    const dim3 grid((B + DEEP_R - 1) / DEEP_R, S);
    for (int l = 1; l < D.L; ++l) {
        const int Hin = D.H[l - 1], Hout = D.H[l];
        const size_t smem = deep_fwd_smem(Hin, Hout);
        if (l == 1 && use_tc) {
            if (int e = deep_smem_attr(bnn_deep_fwd_kernel<true>, smem)) return e;
            bnn_deep_fwd_kernel<true><<<grid, DEEP_THREADS, smem, stream>>>(ws.pre[0], ws.W, D.ldw, D.off[2], D.off[1], B, Hin, Hout,
                                                                            D.act[0], ws.h[0], ws.pre[1]);
        } else {
            if (int e = deep_smem_attr(bnn_deep_fwd_kernel<false>, smem)) return e;
            bnn_deep_fwd_kernel<false><<<grid, DEEP_THREADS, smem, stream>>>(ws.pre[l - 1], ws.W, D.ldw, D.off[2 * l], D.off[2 * l - 1], B,
                                                                             Hin, Hout, D.act[l - 1], ws.h[l - 1], ws.pre[l]);
        }
        BRN_LAUNCH_OK("bnn_deep_fwd_kernel");
    }
    return 0;
}

static int deep_check(const char* fn, const float* X, int B, int P, int n_hidden, const int* H, const int* act, int C,
                      const brn_mf_var* vars, const brn_sample_range* r, bool need_grads, int with_prior) {
    BRN_CHECK_ARG(n_hidden >= 2, "%s: n_hidden=%d; one hidden layer is the two-layer network of brn_bnn_elbo_fwd_bwd_act / "
                  "brn_bnn_predict", fn, n_hidden);
    BRN_CHECK_ARG(n_hidden <= DEEP_MAXL, "%s: n_hidden=%d exceeds the supported maximum %d", fn, n_hidden, DEEP_MAXL);
    BRN_CHECK_ARG(X && H && act && vars && r, "%s: NULL pointer", fn);
    BRN_CHECK_ARG(B > 0 && P > 0 && C > 0, "%s: bad shape B=%d P=%d C=%d", fn, B, P, C);
    BRN_CHECK_ARG(C <= BNN_MAXC, "%s: C=%d exceeds the supported maximum %d", fn, C, BNN_MAXC);
    for (int l = 0; l < n_hidden; ++l) {
        BRN_CHECK_ARG(H[l] > 0 && H[l] <= DEEP_MAXH, "%s: hidden width H[%d]=%d outside [1, %d]", fn, l, H[l], DEEP_MAXH);
        BRN_CHECK_ARG(act[l] >= 0 && act[l] <= 2, "%s: unknown activation act[%d]=%d", fn, l, act[l]);
    }
    if (int e = check_sample_range(*r)) return e;
    const DeepLayout D(B, P, n_hidden, H, act, C);
    for (int v = 0; v < D.nvars(); ++v) {
        BRN_CHECK_ARG(vars[v].numel == D.n[v], "vars[%d].numel=%lld, expected %lld", v, (long long)vars[v].numel, (long long)D.n[v]);
        BRN_CHECK_ARG(vars[v].mu && vars[v].rho, "vars[%d]: NULL parameter pointer", v);
        if (need_grads) {
            BRN_CHECK_ARG(vars[v].dmu && vars[v].drho, "vars[%d]: NULL gradient pointer", v);
            BRN_CHECK_ARG(!with_prior || vars[v].tied || (vars[v].prior_loc && vars[v].prior_scale),
                          "vars[%d]: prior_loc/prior_scale required when not tied", v);
        }
    }
    return 0;
}

}  // namespace brn

using namespace brn;

extern "C" size_t brn_bnn_deep_workspace_bytes(int B, int P, int n_hidden, const int* H, int C, int s_local) {
    if (B <= 0 || P <= 0 || C <= 0 || C > BNN_MAXC || s_local < 0 || !H || n_hidden < 2 || n_hidden > DEEP_MAXL) return 0;
    for (int l = 0; l < n_hidden; ++l)
        if (H[l] <= 0 || H[l] > DEEP_MAXH) return 0;
    return DeepWorkspace(nullptr, DeepLayout(B, P, n_hidden, H, nullptr, C), s_local).bytes;
}

extern "C" int brn_bnn_deep_elbo_fwd_bwd(const float* X, const int32_t* y, int B, int P, int n_hidden, const int* H, const int* act,
                                         int C, const brn_mf_var* vars, const brn_sample_range* r, void* workspace,
                                         size_t workspace_bytes, int with_prior, double* loss, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (int e = deep_check("brn_bnn_deep_elbo_fwd_bwd", X, B, P, n_hidden, H, act, C, vars, r, true, with_prior)) return e;
    BRN_CHECK_ARG(y && loss, "brn_bnn_deep_elbo_fwd_bwd: NULL pointer");
    const char* env_variant = getenv("BRN_BNN_VARIANT");
    BRN_CHECK_ARG(!env_variant || strcmp(env_variant, "tcgen05") || H[0] <= BNN_UMMA_HP,
                  "BRN_BNN_VARIANT=tcgen05 needs H[0] <= %d (got %d)", BNN_UMMA_HP, H[0]);
    const DeepLayout D(B, P, n_hidden, H, act, C);
    const int S = r->s_local, L = D.L, nv = D.nvars();
    if (S == 0) return wait_data_ready(stream);
    const DeepWorkspace ws(workspace, D, S);
    BRN_CHECK_ARG(workspace && workspace_bytes >= ws.bytes, "workspace too small: %zu < %zu", workspace_bytes, ws.bytes);
    const bool use_tc = deep_use_tc(H[0]);
    set_variant(use_tc ? "tcgen05" : "simt");
    if (int e = deep_forward(X, D, vars, r, ws, use_tc, true, stream)) return e;
    {
        StageTimer st("bnn.mid", stream);
        const BnnLayout V = D.head();
        const size_t smem = MidSmem(V.H, C).total * sizeof(float);
        if (int e = deep_smem_attr(bnn_mid2_kernel<false>, smem)) return e;
        bnn_mid2_kernel<false><<<dim3((B + MID_R - 1) / MID_R, S), 256, smem, stream>>>(ws.pre[L - 1], ws.W, ws.dW, y, V,
                                                                                         1.0f / (float)r->s_total, loss, nullptr,
                                                                                         nullptr, 0, 0);
        BRN_LAUNCH_OK("bnn_mid2_kernel");
    }
    {
        StageTimer st("bnn.deep_bwd", stream);
        const dim3 grid((B + DEEP_R - 1) / DEEP_R, S);
        for (int l = L - 1; l >= 1; --l) {
            const int Hin = D.H[l - 1], Hout = D.H[l];
            const size_t smem = deep_bwd_smem(Hin, Hout);
            // dpre_{l-1} replaces pre_{l-1}, which the forward stage l consumed (h_{l-1} is kept)
            if (l == 1 && use_tc) {
                if (int e = deep_smem_attr(bnn_deep_bwd_kernel<true>, smem)) return e;
                bnn_deep_bwd_kernel<true><<<grid, DEEP_THREADS, smem, stream>>>(ws.pre[1], ws.h[0], ws.W, ws.dW, D.ldw, D.off[2], D.off[1], B,
                                                                                Hin, Hout, D.act[0], ws.pre[0], ws.tc.scal + SC_DPRE);
            } else {
                if (int e = deep_smem_attr(bnn_deep_bwd_kernel<false>, smem)) return e;
                bnn_deep_bwd_kernel<false><<<grid, DEEP_THREADS, smem, stream>>>(ws.pre[l], ws.h[l - 1], ws.W, ws.dW, D.ldw, D.off[2 * l],
                                                                                 D.off[2 * l - 1], B, Hin, Hout, D.act[l - 1], ws.pre[l - 1],
                                                                                 nullptr);
            }
            BRN_LAUNCH_OK("bnn_deep_bwd_kernel");
        }
    }
    {
        StageTimer st("bnn.gemm_bwd", stream);
        const int H1 = D.H[0];
        if (use_tc) {
            // dpre_1 has no a-priori bound once W2 is not the head: split it at its measured maximum
            dim3 grid((B + 31) / 32, (BNN_UMMA_HP + 31) / 32, S), block(32, 8);
            bnn_deep_split_dpre_kernel<<<grid, block, 0, stream>>>(ws.pre[0], B, H1, BNN_UMMA_HP, ws.tc.dph, ws.tc.dpl, ws.tc.ldB,
                                                                   ws.tc.scal + SC_DPRE);
            BRN_LAUNCH_OK("bnn_deep_split_dpre_kernel");
            if (int e = bnn_tc_gemm_bwd(B, P, H1, S, D.ldw, ws.tc, ws.dW, ws.tc.scal + SC_DPRE, 1.f, stream)) return e;
        } else if (int e = launch_sgemm_batched<false, false>(ws.pre[0], H1, (int64_t)B * H1, X, P, 0, ws.dW, P, D.ldw, H1, P, B, S,
                                                              stream)) {
            return e;
        }
    }
    StageTimer st("bnn.reduce_finalize", stream);
    for (int v0 = 0; v0 < nv; v0 += 4) {
        const int n = std::min(4, nv - v0);
        int64_t rel[4];
        for (int k = 0; k < n; ++k) rel[k] = D.off[v0 + k] - D.off[v0];
        const int64_t total = D.off[v0 + n - 1] + D.n[v0 + n - 1] - D.off[v0];
        if (int e = launch_mf_reduce_finalize_multi(vars + v0, rel, n, total, ws.eps + D.off[v0], D.ldw, ws.dW + D.off[v0], D.ldw, ws.stats,
                                                    *r, with_prior, loss, stream, 0))
            return e;
    }
    return 0;
}

extern "C" int brn_bnn_deep_predict(const float* X, int B, int P, int n_hidden, const int* H, const int* act, int C,
                                    const brn_mf_var* vars, const brn_sample_range* r, void* workspace, size_t workspace_bytes,
                                    float* logits, int32_t* labels, float* probs_mean, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (int e = deep_check("brn_bnn_deep_predict", X, B, P, n_hidden, H, act, C, vars, r, false, 0)) return e;
    BRN_CHECK_ARG(logits, "brn_bnn_deep_predict: NULL pointer");
    const DeepLayout D(B, P, n_hidden, H, act, C);
    const int S = r->s_local;
    if (S == 0) return 0;
    const DeepWorkspace ws(workspace, D, S);
    BRN_CHECK_ARG(workspace && workspace_bytes >= ws.bytes, "workspace too small: %zu < %zu", workspace_bytes, ws.bytes);
    const bool use_tc = deep_use_tc(H[0]);
    set_variant(use_tc ? "tcgen05" : "simt");
    if (int e = deep_forward(X, D, vars, r, ws, use_tc, false, stream)) return e;
    const BnnLayout V = D.head();
    const size_t smem = sizeof(float) * ((size_t)C * V.H + V.H + C);
    if (int e = deep_smem_attr(bnn_predict_kernel<false>, smem)) return e;
    bnn_predict_kernel<false><<<dim3((B + 127) / 128, S), 128, smem, stream>>>(ws.pre[D.L - 1], ws.W, V, logits, labels, probs_mean,
                                                                               1.0f / (float)r->s_total, *r);
    BRN_LAUNCH_OK("bnn_predict_kernel");
    return 0;
}
