// K3: Bayesian neural network P-H-C (tanh, Categorical likelihood) -- ELBO forward + pathwise backward.
// See include/brancher_cuda.h (brn_bnn_elbo_fwd_bwd) for the contract and the reference lines replaced.
//
// Stage plan (shared by the "simt" and "tcgen05" variants; they differ in stages 2 and 4):
//   1. noise + weight sampling          W_s = mu + softplus(rho) * eps_s                (HBM-bound)
//   2. layer-1 GEMM per sample          pre_s[B,H] = X[B,P] . W1_s^T[P,H]               (GEMM)
//   3. "mid": tanh, layer 2, log-softmax, ll, and backward down to d pre_s              (HBM-bound)
//   4. layer-1 weight gradient          dW1_s[H,P] = dpre_s^T[H,B] . X[B,P]             (GEMM)
//   5. sample-axis reduction + K1a      gw = sum_s dW_s, gwe = sum_s dW_s*eps_s, prior/entropy, chain rule
#include "meanfield.cuh"
#include "sgemm.cuh"
#include "umma_gemm.cuh"
#include <algorithm>
#include <stdlib.h>
#include <type_traits>

namespace brn {

constexpr int BNN_MAXC = 16;

// hidden activation (the matcher accepts BF.tanh / BF.relu / BF.sigmoid): value and derivative, the latter from the
// activation's OUTPUT h, which is all the backward stages keep
constexpr int ACT_TANH = 0, ACT_RELU = 1, ACT_SIGMOID = 2;
__device__ __forceinline__ float act_grad_from_h(int act, float h) {
    return act == ACT_TANH ? __fmaf_rn(-h, h, 1.f) : (act == ACT_RELU ? (h > 0.f ? 1.f : 0.f) : h * (1.f - h));
}
__device__ __forceinline__ float act_exact(int act, float x) {        // SIMT variant / predictive pass: libm accuracy
    return act == ACT_TANH ? tanhf(x) : (act == ACT_RELU ? fmaxf(x, 0.f) : 1.f / (1.f + expf(-x)));
}

struct BnnLayout {
    int B, P, H, C, act;
    int64_t oW1, ob1, oW2, ob2, numel, ldw;
    __host__ __device__ BnnLayout(int B_, int P_, int H_, int C_, int act_ = 0) : B(B_), P(P_), H(H_), C(C_), act(act_) {
        oW1 = 0;
        ob1 = (int64_t)H * P;
        oW2 = ob1 + H;
        ob2 = oW2 + (int64_t)C * H;
        numel = ob2 + C;
        ldw = (numel + 3) / 4 * 4;
    }
};

// One CTA = R rows of the batch for one sample; one thread per row.
// pre (in):  X.W1_s^T without bias;  pre (out): d ll_s / d pre.
// If dpT_hi != NULL the result is written transposed and TF32-split instead of in place:
//   dpT_{hi,lo}[(s*Hp + h) * ldB + b]   (rows h in [H, Hp) zero) -- the K-major B operand of the tcgen05
//   weight-gradient GEMM.
__global__ void bnn_mid_kernel(float* __restrict__ pre, const float* __restrict__ W, float* __restrict__ dW,
                               const int32_t* __restrict__ y, BnnLayout L, int R, float inv_S,
                               double* __restrict__ loss, float* __restrict__ dpT_hi, float* __restrict__ dpT_lo,
                               int Hp, int64_t ldB) {
    extern __shared__ float sm[];
    const int H = L.H, C = L.C, B = L.B, HP = H + 1;
    float* tile = sm;                    // [R][H+1]
    float* W2s = tile + (size_t)R * HP;  // [C][H]
    float* b1s = W2s + C * H;            // [H]
    float* b2s = b1s + H;                // [C]
    float* das = b2s + C;                // [R][C]
    __shared__ double red[32];

    const int s = blockIdx.y, b0 = blockIdx.x * R, t = threadIdx.x, nt = blockDim.x;
    const float* Ws = W + (int64_t)s * L.ldw;
    float* dWs = dW + (int64_t)s * L.ldw;
    float* pre_s = pre + (int64_t)s * B * H;

    if (dpT_hi != nullptr) {     // tcgen05 variant: pre arrives transposed, [S][H][B]
        for (int idx = t; idx < R * H; idx += nt) {
            int h = idx / R, r = idx - h * R;
            tile[r * HP + h] = (b0 + r < B) ? pre_s[(int64_t)h * B + b0 + r] : 0.f;
        }
    } else {
        for (int idx = t; idx < R * H; idx += nt) {
            int r = idx / H, h = idx - r * H;
            tile[r * HP + h] = (b0 + r < B) ? pre_s[(int64_t)(b0 + r) * H + h] : 0.f;
        }
    }
    for (int idx = t; idx < C * H; idx += nt) W2s[idx] = Ws[L.oW2 + idx];
    for (int idx = t; idx < H; idx += nt) b1s[idx] = Ws[L.ob1 + idx];
    for (int idx = t; idx < C; idx += nt) b2s[idx] = Ws[L.ob2 + idx];
    __syncthreads();

    const int r = t;
    const bool valid = (r < R) && (b0 + r < B);
    float da[BNN_MAXC];
    float ll = 0.f;
    if (valid) {
        float a[BNN_MAXC];
#pragma unroll
        for (int c = 0; c < BNN_MAXC; ++c) a[c] = 0.f;
        for (int h = 0; h < H; ++h) {
            float v = act_exact(L.act, tile[r * HP + h] + b1s[h]);
            tile[r * HP + h] = v;
#pragma unroll
            for (int c = 0; c < BNN_MAXC; ++c)
                if (c < C) a[c] = __fmaf_rn(W2s[c * H + h], v, a[c]);
        }
        float m = -INFINITY;
#pragma unroll
        for (int c = 0; c < BNN_MAXC; ++c)
            if (c < C) { a[c] += b2s[c]; m = fmaxf(m, a[c]); }
        float se = 0.f;
#pragma unroll
        for (int c = 0; c < BNN_MAXC; ++c)
            if (c < C) se += expf(a[c] - m);
        const float lse = m + logf(se);
        const int label = y[b0 + r];
#pragma unroll
        for (int c = 0; c < BNN_MAXC; ++c) {
            if (c < C) {
                float p = expf(a[c] - lse);
                da[c] = (c == label ? 1.f : 0.f) - p;      // d ll / d a_c
                if (c == label) ll = a[c] - lse;
            } else da[c] = 0.f;
        }
    } else {
#pragma unroll
        for (int c = 0; c < BNN_MAXC; ++c) da[c] = 0.f;
    }
    if (r < R)
        for (int c = 0; c < C; ++c) das[r * C + c] = da[c];
    __syncthreads();

    // dW2_s[c,h] += sum_r da_r[c] * h_r[h] ;  db2_s[c] += sum_r da_r[c]
    for (int o = t; o < C * H; o += nt) {
        int c = o / H, h = o - c * H;
        float acc = 0.f;
        for (int rr = 0; rr < R; ++rr) acc = __fmaf_rn(das[rr * C + c], tile[rr * HP + h], acc);
        atomicAdd(&dWs[L.oW2 + o], acc);
    }
    for (int c = t; c < C; c += nt) {
        float acc = 0.f;
        for (int rr = 0; rr < R; ++rr) acc += das[rr * C + c];
        atomicAdd(&dWs[L.ob2 + c], acc);
    }
    __syncthreads();

    if (r < R) {
        for (int h = 0; h < H; ++h) {
            float hv = tile[r * HP + h];
            float dh = 0.f;
#pragma unroll
            for (int c = 0; c < BNN_MAXC; ++c)
                if (c < C) dh = __fmaf_rn(da[c], W2s[c * H + h], dh);
            tile[r * HP + h] = dh * act_grad_from_h(L.act, hv);
        }
    }
    __syncthreads();

    for (int h = t; h < H; h += nt) {
        float acc = 0.f;
        for (int rr = 0; rr < R; ++rr) acc += tile[rr * HP + h];
        atomicAdd(&dWs[L.ob1 + h], acc);
    }
    if (dpT_hi != nullptr) {
        for (int idx = t; idx < Hp * R; idx += nt) {
            int h = idx / R, rr = idx - h * R;
            if (b0 + rr >= B) continue;
            float hi = 0.f, lo = 0.f;
            if (h < H) umma::split_tf32(tile[rr * HP + h], hi, lo);
            int64_t o = ((int64_t)s * Hp + h) * ldB + b0 + rr;
            dpT_hi[o] = hi;
            dpT_lo[o] = lo;
        }
    } else {
        for (int idx = t; idx < R * H; idx += nt) {
            int rr = idx / H, h = idx - rr * H;
            if (b0 + rr < B) pre_s[(int64_t)(b0 + rr) * H + h] = tile[rr * HP + h];
        }
    }
    double tot = block_sum<double>((double)ll, red);
    if (t == 0) atomicAdd(loss, -tot * (double)inv_S);
}

// ---------------------------------------------------------------------------------------------------
// "mid" stage, fast version: one CTA = 128 batch rows of one sample, 256 threads = 2 threads per row (each owns
// half of the hidden units).  Everything between the two layer-1 GEMMs happens here in shared memory:
//   h = tanh(pre + b1), a = W2 h + b2, log-softmax, ll, da, dW2 / db2 (reduced over the 128 rows),
//   dh = W2^T da, dpre = dh (1 - h^2), db1.
// TC: `pre` arrives transposed [S][H][B] (tcgen05 GEMM output) and dpre leaves transposed + TF32-split
// ([S*Hp][ldB] hi/lo, rows h >= H zero), both coalesced along the batch axis; else `pre` is [S][B][H] and is
// overwritten in place.
// ---------------------------------------------------------------------------------------------------
constexpr int MID_R = 128;

struct MidSmem {
    int HP1;              // odd row pitch of the tile -> conflict-free column and row access
    size_t tile, w2, b1, b2, das, apart, total;   // offsets in floats
    __host__ __device__ MidSmem(int H, int C) {
        HP1 = H | 1;
        tile = 0;
        w2 = tile + (size_t)MID_R * HP1;
        b1 = w2 + (size_t)C * H;
        b2 = b1 + H;
        das = (b2 + C + 3) / 4 * 4;          // float4-aligned
        apart = das + MID_R * 16;
        total = apart + MID_R * 16;
    }
};

template <bool TC>
__global__ void __launch_bounds__(256)
bnn_mid2_kernel(float* __restrict__ pre, const float* __restrict__ W, float* __restrict__ dW,
                const int32_t* __restrict__ y, BnnLayout L, float inv_S, double* __restrict__ loss,
                float* __restrict__ dpT_hi, float* __restrict__ dpT_lo, int Hp, int64_t ldB) {
    extern __shared__ __align__(16) float sm[];
    const int H = L.H, C = L.C, B = L.B;
    const MidSmem M(H, C);
    const int HP1 = M.HP1;
    float* tile = sm + M.tile;
    float* W2s = sm + M.w2;
    float* b1s = sm + M.b1;
    float* b2s = sm + M.b2;
    float* das = sm + M.das;      // [128][16]
    float* apart = sm + M.apart;  // [128][16]
    __shared__ double red[32];

    const int s = blockIdx.y, b0 = blockIdx.x * MID_R, t = threadIdx.x;
    const int r = t & (MID_R - 1), half = t >> 7;
    const float* Ws = W + (int64_t)s * L.ldw;
    float* dWs = dW + (int64_t)s * L.ldw;
    float* pre_s = pre + (int64_t)s * B * H;
    const bool row_ok = b0 + r < B;

    // ---- P0: stage the tile
    if (TC) {
        for (int h = half; h < H; h += 2) tile[r * HP1 + h] = row_ok ? pre_s[(int64_t)h * B + b0 + r] : 0.f;
    } else {
        for (int idx = t; idx < MID_R * H; idx += 256) {
            int rr = idx / H, h = idx - rr * H;
            tile[rr * HP1 + h] = (b0 + rr < B) ? pre_s[(int64_t)(b0 + rr) * H + h] : 0.f;
        }
    }
    for (int idx = t; idx < C * H; idx += 256) W2s[idx] = Ws[L.oW2 + idx];
    for (int idx = t; idx < H; idx += 256) b1s[idx] = Ws[L.ob1 + idx];
    for (int idx = t; idx < C; idx += 256) b2s[idx] = Ws[L.ob2 + idx];
    __syncthreads();

    // ---- P1: hidden activations + logits (each thread: its half of the hidden units)
    const int Hh = (H + 1) >> 1, h0 = half * Hh, h1 = min(H, h0 + Hh);
    float a[BNN_MAXC];
#pragma unroll
    for (int c = 0; c < BNN_MAXC; ++c) a[c] = 0.f;
    for (int h = h0; h < h1; ++h) {
        float v = act_exact(L.act, tile[r * HP1 + h] + b1s[h]);
        tile[r * HP1 + h] = v;
#pragma unroll
        for (int c = 0; c < BNN_MAXC; ++c)
            if (c < C) a[c] = __fmaf_rn(W2s[c * H + h], v, a[c]);
    }
    if (half == 1) {
#pragma unroll
        for (int c = 0; c < BNN_MAXC; ++c) apart[r * 16 + c] = a[c];
    }
    __syncthreads();
    float da[BNN_MAXC];
    float ll = 0.f;
    if (half == 0) {
        if (row_ok) {
            float m = -INFINITY;
#pragma unroll
            for (int c = 0; c < BNN_MAXC; ++c)
                if (c < C) { a[c] += apart[r * 16 + c] + b2s[c]; m = fmaxf(m, a[c]); }
            float se = 0.f;
#pragma unroll
            for (int c = 0; c < BNN_MAXC; ++c)
                if (c < C) se += expf(a[c] - m);
            const float lse = m + logf(se);
            const int label = y[b0 + r];
#pragma unroll
            for (int c = 0; c < BNN_MAXC; ++c) {
                if (c < C) {
                    da[c] = (c == label ? 1.f : 0.f) - expf(a[c] - lse);      // d ll / d a_c
                    if (c == label) ll = a[c] - lse;
                } else da[c] = 0.f;
            }
        } else {
#pragma unroll
            for (int c = 0; c < BNN_MAXC; ++c) da[c] = 0.f;
        }
#pragma unroll
        for (int c = 0; c < BNN_MAXC; ++c) das[r * 16 + c] = da[c];
    }
    __syncthreads();

    // ---- P2: dW2_s[c,h] += sum_r da_r[c] h_r[h] ; db2_s[c] += sum_r da_r[c]
    {
        const int g = half;                           // class group: classes [8g, 8g+8)
        if (8 * g < C) {
            for (int hh = r; hh < H; hh += MID_R) {
                float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
                for (int rr = 0; rr < MID_R; ++rr) {
                    const float hv = tile[rr * HP1 + hh];
                    const float4 d0 = *reinterpret_cast<const float4*>(&das[rr * 16 + 8 * g]);
                    const float4 d1 = *reinterpret_cast<const float4*>(&das[rr * 16 + 8 * g + 4]);
                    acc[0] = __fmaf_rn(d0.x, hv, acc[0]); acc[1] = __fmaf_rn(d0.y, hv, acc[1]);
                    acc[2] = __fmaf_rn(d0.z, hv, acc[2]); acc[3] = __fmaf_rn(d0.w, hv, acc[3]);
                    acc[4] = __fmaf_rn(d1.x, hv, acc[4]); acc[5] = __fmaf_rn(d1.y, hv, acc[5]);
                    acc[6] = __fmaf_rn(d1.z, hv, acc[6]); acc[7] = __fmaf_rn(d1.w, hv, acc[7]);
                }
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    if (8 * g + j < C) atomicAdd(&dWs[L.oW2 + (int64_t)(8 * g + j) * H + hh], acc[j]);
            }
        }
        if (t < C) {
            float acc = 0.f;
            for (int rr = 0; rr < MID_R; ++rr) acc += das[rr * 16 + t];
            atomicAdd(&dWs[L.ob2 + t], acc);
        }
    }
    __syncthreads();

    // ---- P3: dpre = (W2^T da) (1 - h^2)
    if (half == 1) {
#pragma unroll
        for (int c = 0; c < BNN_MAXC; ++c) da[c] = das[r * 16 + c];
    }
    for (int h = h0; h < h1; ++h) {
        const float hv = tile[r * HP1 + h];
        float dh = 0.f;
#pragma unroll
        for (int c = 0; c < BNN_MAXC; ++c)
            if (c < C) dh = __fmaf_rn(da[c], W2s[c * H + h], dh);
        tile[r * HP1 + h] = dh * act_grad_from_h(L.act, hv);
    }
    __syncthreads();

    // ---- P4: db1_s[h] += sum_r dpre_r[h] ; write dpre
    for (int hh = r; hh < H; hh += MID_R) {
        float acc = 0.f;
        const int r0 = half * (MID_R / 2);
#pragma unroll 8
        for (int rr = r0; rr < r0 + MID_R / 2; ++rr) acc += tile[rr * HP1 + hh];
        atomicAdd(&dWs[L.ob1 + hh], acc);
    }
    if (TC) {
        if (row_ok) {
            for (int h = half; h < Hp; h += 2) {
                float hi = 0.f, lo = 0.f;
                if (h < H) umma::split_tf32(tile[r * HP1 + h], hi, lo);
                const int64_t o = ((int64_t)s * Hp + h) * ldB + b0 + r;
                dpT_hi[o] = hi;
                dpT_lo[o] = lo;
            }
        }
    } else {
        for (int idx = t; idx < MID_R * H; idx += 256) {
            int rr = idx / H, h = idx - rr * H;
            if (b0 + rr < B) pre_s[(int64_t)(b0 + rr) * H + h] = tile[rr * HP1 + h];
        }
    }
    double tot = block_sum<double>((double)ll, red);
    if (t == 0) atomicAdd(loss, -tot * (double)inv_S);
}


// ---------------------------------------------------------------------------------------------------
// posterior-predictive forward pass (SURVEY 8(f)3): logits of every (posterior sample, data row) in one launch, optional
// class draws (inverse CDF on a Philox uniform) and the MC average of the class probabilities.
// One CTA = 128 rows of one sample, one thread per row.  PRE_T: pre is [S][H][B] (tcgen05 variant) else [S][B][H].
// ---------------------------------------------------------------------------------------------------
template <bool PRE_T>
__global__ void __launch_bounds__(128)
bnn_predict_kernel(const float* __restrict__ pre, const float* __restrict__ W, BnnLayout L, float* __restrict__ logits,
                   int32_t* __restrict__ labels, float* __restrict__ probs_mean, float inv_S, brn_sample_range r) {
    extern __shared__ float sm[];
    const int H = L.H, C = L.C, B = L.B;
    float* W2s = sm;                 // [C][H]
    float* b1s = W2s + C * H;        // [H]
    float* b2s = b1s + H;            // [C]
    const int s = blockIdx.y, b = blockIdx.x * 128 + threadIdx.x;
    const float* Ws = W + (int64_t)s * L.ldw;
    for (int i = threadIdx.x; i < C * H; i += 128) W2s[i] = Ws[L.oW2 + i];
    for (int i = threadIdx.x; i < H; i += 128) b1s[i] = Ws[L.ob1 + i];
    for (int i = threadIdx.x; i < C; i += 128) b2s[i] = Ws[L.ob2 + i];
    __syncthreads();
    if (b >= B) return;
    const float* ps = pre + (int64_t)s * B * H;
    float a[BNN_MAXC];
#pragma unroll
    for (int c = 0; c < BNN_MAXC; ++c) a[c] = 0.f;
    for (int h = 0; h < H; ++h) {
        const float v = act_exact(L.act, (PRE_T ? ps[(int64_t)h * B + b] : ps[(int64_t)b * H + h]) + b1s[h]);
#pragma unroll
        for (int c = 0; c < BNN_MAXC; ++c)
            if (c < C) a[c] = __fmaf_rn(W2s[c * H + h], v, a[c]);
    }
    float m = -INFINITY;
#pragma unroll
    for (int c = 0; c < BNN_MAXC; ++c)
        if (c < C) { a[c] += b2s[c]; m = fmaxf(m, a[c]); }
    float* lo = logits + ((int64_t)s * B + b) * C;
    float se = 0.f, e[BNN_MAXC];
#pragma unroll
    for (int c = 0; c < BNN_MAXC; ++c)
        if (c < C) { lo[c] = a[c]; e[c] = expf(a[c] - m); se += e[c]; }
    const float inv = 1.f / se;
    if (probs_mean) {
#pragma unroll
        for (int c = 0; c < BNN_MAXC; ++c)
            if (c < C) atomicAdd(&probs_mean[(int64_t)b * C + c], e[c] * inv * inv_S);
    }
    if (labels) {      // k ~ Categorical(logits) (distributions.py:275-311): inverse CDF on one Philox uniform per (sample, row)
        const Philox4 u4 = philox4x32_10((uint32_t)(b >> 2), (uint32_t)(r.s0 + s), 4u, (uint32_t)philox_offset(r), (uint32_t)r.seed,
                                         (uint32_t)(r.seed >> 32) ^ (uint32_t)(philox_offset(r) >> 32));
        const uint32_t w = (b & 3) == 0 ? u4.x : ((b & 3) == 1 ? u4.y : ((b & 3) == 2 ? u4.z : u4.w));
        const float u = u01(w) * se;
        float acc = 0.f;
        int k = C - 1;
#pragma unroll
        for (int c = 0; c < BNN_MAXC; ++c)
            if (c < C) { acc += e[c]; if (u <= acc && k == C - 1 && c < C - 1) k = c; }
        labels[(int64_t)s * B + b] = k;
    }
}

static size_t bnn_mid_smem(int R, int H, int C) {
    return sizeof(float) * ((size_t)R * (H + 1) + (size_t)C * H + H + C + (size_t)R * C);
}

}  // namespace brn
#include "bnn_tc.cuh"
namespace brn {

struct BnnWorkspace {
    float *eps, *W, *dW, *pre, *stats;
    BnnTcWorkspace tc;
    size_t bytes;
    BnnWorkspace(void* base, const BnnLayout& L, int S) {
        WorkspaceCarver take(base);
        eps = take((size_t)S * L.ldw);
        W = take((size_t)S * L.ldw);
        dW = take((size_t)S * L.ldw);
        pre = take((size_t)S * L.B * L.H);
        stats = take(4 * (size_t)L.ldw);
        tc.carve(take, L, S);
        bytes = take.off;
    }
};

}  // namespace brn

using namespace brn;

extern "C" size_t brn_bnn_workspace_bytes(int B, int P, int H, int C, int s_local) {
    if (B <= 0 || P <= 0 || H <= 0 || C <= 0 || s_local < 0) return 0;
    BnnLayout L(B, P, H, C);
    return BnnWorkspace(nullptr, L, s_local).bytes;
}

extern "C" int brn_bnn_elbo_fwd_bwd(const float* X, const int32_t* y, int B, int P, int H, int C,
                                    const brn_mf_var vars[4], const brn_sample_range* r, void* workspace,
                                    size_t workspace_bytes, int with_prior, double* loss, void* stream_) {
    return brn_bnn_elbo_fwd_bwd_act(X, y, B, P, H, C, BRN_ACT_TANH, vars, r, workspace, workspace_bytes, with_prior, loss, stream_);
}

extern "C" int brn_bnn_elbo_fwd_bwd_act(const float* X, const int32_t* y, int B, int P, int H, int C, int activation,
                                        const brn_mf_var vars[4], const brn_sample_range* r, void* workspace,
                                        size_t workspace_bytes, int with_prior, double* loss, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    BRN_CHECK_ARG(X && y && vars && r && loss, "brn_bnn_elbo_fwd_bwd: NULL pointer");
    BRN_CHECK_ARG(activation >= 0 && activation <= 2, "brn_bnn_elbo_fwd_bwd: unknown activation %d", activation);
    BRN_CHECK_ARG(B > 0 && P > 0 && H > 0 && C > 0, "brn_bnn_elbo_fwd_bwd: bad shape B=%d P=%d H=%d C=%d", B, P, H, C);
    BRN_CHECK_ARG(C <= BNN_MAXC, "brn_bnn_elbo_fwd_bwd: C=%d exceeds the supported maximum %d", C, BNN_MAXC);
    if (int e = check_sample_range(*r)) return e;
    BnnLayout L(B, P, H, C, activation);
    const int64_t numels[4] = {(int64_t)H * P, H, (int64_t)C * H, C};
    const int64_t offs[4] = {L.oW1, L.ob1, L.oW2, L.ob2};
    for (int v = 0; v < 4; ++v) {
        BRN_CHECK_ARG(vars[v].numel == numels[v], "vars[%d].numel=%lld, expected %lld", v, (long long)vars[v].numel,
                      (long long)numels[v]);
        BRN_CHECK_ARG(vars[v].mu && vars[v].rho && vars[v].dmu && vars[v].drho, "vars[%d]: NULL parameter pointer", v);
        BRN_CHECK_ARG(!with_prior || vars[v].tied || (vars[v].prior_loc && vars[v].prior_scale),
                      "vars[%d]: prior_loc/prior_scale required when not tied", v);
    }
    const int S = r->s_local;
    if (S == 0) return wait_data_ready((cudaStream_t)stream_);
    BnnWorkspace ws(workspace, L, S);
    BRN_CHECK_ARG(workspace && workspace_bytes >= ws.bytes, "workspace too small: %zu < %zu", workspace_bytes, ws.bytes);
    // variant: tcgen05 (TMA + 3xFP16 tensor-core GEMMs) when the padded hidden width matches the instantiated
    // tile, else the fp32 SIMT GEMMs.  BRN_BNN_VARIANT=simt|tcgen05 forces one (tests compare both).
    const char* env_variant = getenv("BRN_BNN_VARIANT");
    bool use_tc = (H > BNN_UMMA_HP - 16 && H <= BNN_UMMA_HP);
    if (env_variant) {
        if (!strcmp(env_variant, "simt")) use_tc = false;
        else if (!strcmp(env_variant, "tcgen05")) {
            BRN_CHECK_ARG(H <= BNN_UMMA_HP, "BRN_BNN_VARIANT=tcgen05 needs H <= %d (got %d)", BNN_UMMA_HP, H);
            use_tc = true;
        }
    }
    set_variant(use_tc ? "tcgen05" : "simt");
    if (use_tc) return bnn_tc_eval(X, y, L, vars, r, ws.tc, ws.eps, ws.W, ws.dW, ws.pre, ws.stats, with_prior, loss, stream);

    // ---- SIMT variant
    // 1. noise + weights: noise in ws.eps [S][ldw], sampled weights in ws.W, the four variables back to back inside a row
    {
        StageTimer st("bnn.sample_weights", stream);
        if (int e = launch_sample_multi(vars, offs, 4, ws.eps, ws.W, L.ldw, *r, stream)) return e;
        if (int e = wait_data_ready(stream)) return e;
    }
    // 2. pre_s = X . W1_s^T
    {
        StageTimer st("bnn.gemm_fwd", stream);
        if (int e = launch_sgemm_batched<true, true>(X, P, 0, ws.W + L.oW1, P, L.ldw, ws.pre, H, (int64_t)B * H, B, H, P, S, stream))
            return e;
    }
    // 3. mid
    BRN_CUDA_OK(cudaMemset2DAsync(ws.dW + L.ob1, L.ldw * sizeof(float), 0, (L.numel - L.ob1) * sizeof(float), S, stream));
    {
        StageTimer st("bnn.mid", stream);
        const float inv_S = 1.0f / (float)r->s_total;
        const MidSmem ms(H, C);
        const size_t smem2 = ms.total * sizeof(float);
        if (smem2 <= 200 * 1024) {
            dim3 grid((B + MID_R - 1) / MID_R, S);
            BRN_CUDA_OK(cudaFuncSetAttribute(bnn_mid2_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2));
            bnn_mid2_kernel<false><<<grid, 256, smem2, stream>>>(ws.pre, ws.W, ws.dW, y, L, inv_S, loss, nullptr, nullptr, 0, 0);
            BRN_LAUNCH_OK("bnn_mid2_kernel");
        } else {
            // very wide hidden layers: the one-thread-per-row kernel with fewer rows per CTA
            int R = 128;
            while (R > 32 && bnn_mid_smem(R, H, C) > 200 * 1024) R -= 32;
            size_t smem = bnn_mid_smem(R, H, C);
            BRN_CHECK_ARG(smem <= 220 * 1024, "brn_bnn_elbo_fwd_bwd: hidden width H=%d too large for the mid kernel", H);
            BRN_CUDA_OK(cudaFuncSetAttribute(bnn_mid_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            dim3 grid((B + R - 1) / R, S);
            bnn_mid_kernel<<<grid, R, smem, stream>>>(ws.pre, ws.W, ws.dW, y, L, R, inv_S, loss, nullptr, nullptr, 0, 0);
            BRN_LAUNCH_OK("bnn_mid_kernel");
        }
    }
    // 4. dW1_s = dpre_s^T . X
    {
        StageTimer st("bnn.gemm_bwd", stream);
        if (int e = launch_sgemm_batched<false, false>(ws.pre, H, (int64_t)B * H, X, P, 0, ws.dW + L.oW1, P, L.ldw, H, P, B, S, stream))
            return e;
    }
    // 5. reduce over samples + prior/entropy + chain rule: one stats launch for all four variables
    StageTimer st5("bnn.reduce_finalize", stream);
    return launch_mf_reduce_finalize_multi(vars, offs, 4, L.numel, ws.eps, L.ldw, ws.dW, L.ldw, ws.stats, *r, with_prior, loss, stream, 0);
}

extern "C" int brn_bnn_predict(const float* X, int B, int P, int H, int C, int activation, const brn_mf_var vars[4],
                               const brn_sample_range* r, void* workspace, size_t workspace_bytes, float* logits, int32_t* labels,
                               float* probs_mean, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    BRN_CHECK_ARG(activation >= 0 && activation <= 2, "brn_bnn_predict: unknown activation %d", activation);
    BRN_CHECK_ARG(X && vars && r && logits, "brn_bnn_predict: NULL pointer");
    BRN_CHECK_ARG(B > 0 && P > 0 && H > 0 && C > 0 && C <= BNN_MAXC, "brn_bnn_predict: bad shape B=%d P=%d H=%d C=%d", B, P, H, C);
    if (int e = check_sample_range(*r)) return e;
    BnnLayout L(B, P, H, C, activation);
    const int64_t numels[4] = {(int64_t)H * P, H, (int64_t)C * H, C};
    const int64_t offs[4] = {L.oW1, L.ob1, L.oW2, L.ob2};
    for (int v = 0; v < 4; ++v) {
        BRN_CHECK_ARG(vars[v].numel == numels[v], "vars[%d].numel=%lld, expected %lld", v, (long long)vars[v].numel, (long long)numels[v]);
        BRN_CHECK_ARG(vars[v].mu && vars[v].rho, "vars[%d]: NULL parameter pointer", v);
    }
    const int S = r->s_local;
    if (S == 0) return 0;
    BnnWorkspace ws(workspace, L, S);
    BRN_CHECK_ARG(workspace && workspace_bytes >= ws.bytes, "workspace too small: %zu < %zu", workspace_bytes, ws.bytes);
    const char* env_variant = getenv("BRN_BNN_VARIANT");
    bool use_tc = (H > BNN_UMMA_HP - 16 && H <= BNN_UMMA_HP);
    if (env_variant) {
        if (!strcmp(env_variant, "simt")) use_tc = false;
        else if (!strcmp(env_variant, "tcgen05") && H <= BNN_UMMA_HP) use_tc = true;
    }
    set_variant(use_tc ? "tcgen05" : "simt");
    if (use_tc) {
        if (int e = bnn_tc_eval(X, nullptr, L, vars, r, ws.tc, ws.eps, ws.W, ws.dW, ws.pre, ws.stats, 0, nullptr, stream, true))
            return e;
    } else {
        if (int e = launch_sample_multi(vars, offs, 4, ws.eps, ws.W, L.ldw, *r, stream)) return e;
        if (int e = launch_sgemm_batched<true, true>(X, P, 0, ws.W + L.oW1, P, L.ldw, ws.pre, H, (int64_t)B * H, B, H, P, S, stream))
            return e;
    }
    const size_t smem = sizeof(float) * ((size_t)C * H + H + C);
    BRN_CHECK_ARG(smem <= 200 * 1024, "brn_bnn_predict: hidden width H=%d too large", H);
    dim3 grid((B + 127) / 128, S);
    const float inv_S = 1.0f / (float)r->s_total;
    if (use_tc) {
        BRN_CUDA_OK(cudaFuncSetAttribute(bnn_predict_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        bnn_predict_kernel<true><<<grid, 128, smem, stream>>>(ws.pre, ws.W, L, logits, labels, probs_mean, inv_S, *r);
    } else {
        BRN_CUDA_OK(cudaFuncSetAttribute(bnn_predict_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        bnn_predict_kernel<false><<<grid, 128, smem, stream>>>(ws.pre, ws.W, L, logits, labels, probs_mean, inv_S, *r);
    }
    BRN_LAUNCH_OK("bnn_predict_kernel");
    return 0;
}

#include "bnn_deep.cuh"
