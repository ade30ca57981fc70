// K3 on the tensor cores (tcgen05 + TMA): everything of brn_bnn_elbo_fwd_bwd's "tcgen05" variant.  Included by bnn.cu.
//
// Operand format: "3xFP16".  Both GEMM operands are split into fp16 (hi, lo) pairs -- hi = rn_fp16(x), lo = rn_fp16(x - hi):
// 11 + 11 mantissa bits, exactly what the TF32 (hi, lo) pair of the 3xTF32 scheme carries -- and the three products
// A_lo.B_hi + A_hi.B_lo + A_hi.B_hi run as tcgen05.mma kind::f16 with fp32 accumulation: twice the MACs per instruction and
// half the operand bytes (HBM, L2, shared memory) of kind::tf32.  fp16 has 5 exponent bits, so every operand tensor is
// multiplied by a power of two (exact) that puts its largest magnitude in [2^13, 2^14); the epilogues divide the accumulator
// by the two powers.  The bounds come from the device, no host synchronisation:
//     scal[0] = max_i |mu1_i| + E sigma1_i   (>= |W1_s| for every sample)     scal[2] = max |X|
//     scal[1] = max_i |mu2_i| + E sigma2_i   (dpre = (W2^T da)(1 - h^2), sum_c |da_c| <= 2  =>  |dpre| <= 2 scal[1])
//     scal[3] = max |injected eps| (0 for Philox noise, whose Box-Muller normals are bounded by sqrt(50 ln 2) < 5.9)
// Elements far below the tensor maximum lose RELATIVE precision once their lo part becomes an fp16 subnormal (absolute
// error <= 2^-25 on the scaled tensor, i.e. 2^-38 of the maximum): invisible in a dot product.
#pragma once
#include <cuda_fp16.h>
#include "meanfield.cuh"
#include "umma_gemm.cuh"

namespace brn {

constexpr int SC_W1 = 0, SC_W2 = 1, SC_X = 2, SC_EPS = 3, SC_SLOTS = 16;
constexpr float PHILOX_EPS_MAX = 6.0f;

__device__ __forceinline__ float w1_scale(const float* scal) { return p2_scale(scal[SC_W1]); }
__device__ __forceinline__ float x_scale(const float* scal) { return p2_scale(scal[SC_X]); }
__device__ __forceinline__ float dpre_scale(const float* scal) { return p2_scale(2.f * scal[SC_W2]); }
__device__ __forceinline__ void split_f16(float x, __half& hi, __half& lo) {
    hi = __float2half_rn(x);
    lo = __float2half_rn(x - __half2float(hi));
}
__device__ __forceinline__ void atomic_absmax(float* slot, float v) {        // v >= 0: the uint order is the float order
    atomicMax(reinterpret_cast<unsigned int*>(slot), __float_as_uint(v));
}

// block-wide max of non-negative values -> ONE atomic per block (thousands of same-address atomics cost more than the pass)
__device__ __forceinline__ void block_absmax_to(float m, float* slot) {
    __shared__ float red[8];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = red[0];
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) t = fmaxf(t, red[w]);
        if (t > 0.f) atomic_absmax(slot, t);
    }
    __syncthreads();
}

__global__ void __launch_bounds__(256) absmax_kernel(const float* __restrict__ x, int64_t n, float* __restrict__ slot) {
    float m = 0.f;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if ((reinterpret_cast<uintptr_t>(x) & 15) == 0) {           // 16-byte loads over the aligned body
        const float4* x4 = reinterpret_cast<const float4*>(x);
        for (int64_t q = i; q < n / 4; q += stride) {
            const float4 v = __ldg(x4 + q);
            m = fmaxf(fmaxf(m, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
        }
        for (int64_t j = n / 4 * 4 + i; j < n; j += stride) m = fmaxf(m, fabsf(x[j]));
    } else {
        for (; i < n; i += stride) m = fmaxf(m, fabsf(x[i]));
    }
    block_absmax_to(m, slot);
}
static int launch_absmax(const float* x, int64_t n, float* slot, cudaStream_t stream) {
    if (n <= 0) return 0;
    const unsigned grid = (unsigned)std::min<int64_t>((n / 4 + 255) / 256 + 1, 592);
    absmax_kernel<<<grid, 256, 0, stream>>>(x, n, slot);
    BRN_LAUNCH_OK("absmax_kernel");
    return 0;
}

// scal[SC_W1], scal[SC_W2] = max_i |mu_i| + E softplus(rho_i) over the two weight matrices (one launch)
__global__ void __launch_bounds__(256)
bnn_bounds_kernel(const float* __restrict__ mu1, const float* __restrict__ rho1, int64_t n1, const float* __restrict__ mu2,
                  const float* __restrict__ rho2, int64_t n2, float* __restrict__ scal) {
    const float E = fmaxf(PHILOX_EPS_MAX, scal[SC_EPS]);
    float m1 = 0.f, m2 = 0.f;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n1 + n2; i += (int64_t)gridDim.x * blockDim.x) {
        if (i < n1) m1 = fmaxf(m1, fabsf(mu1[i]) + E * softplusf(rho1[i]));
        else m2 = fmaxf(m2, fabsf(mu2[i - n1]) + E * softplusf(rho2[i - n1]));
    }
    block_absmax_to(m1, scal + SC_W1);
    block_absmax_to(m2, scal + SC_W2);
}

// X [rows][cols] fp32 -> fp16 (hi, lo) pairs scaled by x_scale: row-major [rows][ldd] and transposed [cols][ldt]
__global__ void split_f16_kernel(const float* __restrict__ src, int64_t lds, int rows, int cols, __half* __restrict__ hi,
                                 __half* __restrict__ lo, int64_t ldd, __half* __restrict__ thi, __half* __restrict__ tlo,
                                 int64_t ldt, const float* __restrict__ scal) {
    __shared__ __half th[32][34], tl[32][34];
    const float sc = x_scale(scal);
    const int c0 = blockIdx.y * 32, r0 = blockIdx.x * 32;
    const int tx = threadIdx.x, ty = threadIdx.y;       // 32 x 8
    for (int i = ty; i < 32; i += 8) {
        const int r = r0 + i, c = c0 + tx;
        __half h = __float2half_rn(0.f), l = h;
        if (r < rows && c < cols) {
            split_f16(src[(int64_t)r * lds + c] * sc, h, l);
            hi[(int64_t)r * ldd + c] = h;
            lo[(int64_t)r * ldd + c] = l;
        }
        th[i][tx] = h; tl[i][tx] = l;
    }
    __syncthreads();
    for (int i = ty; i < 32; i += 8) {
        const int c = c0 + i, r = r0 + tx;
        if (r < rows && c < cols) {
            thi[(int64_t)c * ldt + r] = th[tx][i];
            tlo[(int64_t)c * ldt + r] = tl[tx][i];
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// "mid" stage of the tcgen05 variant on the warp-level tensor cores (mma.sync m16n8k8 tf32, 3xTF32 split): the three
// small per-sample contractions of layer 2 are matrix products with one tiny dimension (C <= 16),
//   A  a[b, c]    = sum_h h[b, h] W2[c, h]           M = rows,  N = 16 classes, K = HP hidden
//   B  dh[b, h]   = sum_c da[b, c] W2[c, h]          M = rows,  N = HP hidden,  K = 16 classes
//   C  dW2[c, h]  = sum_b da[b, c] h[b, h]           M = 16 classes, N = HP hidden, K = 128 rows
// and cost ~10 k thread instructions per row as scalar FMAs (issue-bound, 140 us at C3).  Here one CTA
// = 128 batch rows of one sample, 8 warps, warp w = rows [16w, 16w+16) = one MMA m-tile.  The fragment layouts are
// chained without any shuffles by permuting the contraction index: the k-columns (t, t+4) of an A fragment are mapped
// to the consecutive pair (2t, 2t+1) of hidden units (phase A) / classes (phase B), which is exactly how the C fragment
// of the previous product holds them.  Only phase C needs transposed operands and goes through shared memory
// (tile[h][b] pitch 132, das[b][c] pitch 24: both conflict-free for the fragment loads).
// Accuracy: fp32-equivalent via the 3-product split; the hi*hi products and the two correction products accumulate in
// separate chains of at most 16 MMAs.
// ---------------------------------------------------------------------------------------------------
constexpr int MID4_R = 128, MID4_TP = 132, MID4_DP = 24, MID4_THREADS = 256;

template <int HP>
struct Mid4Smem {
    static constexpr int KS = HP / 8;
    // offsets in floats (all multiples of 4)
    static constexpr size_t fragA = 0;                                    // [KS][2][32] float4
    static constexpr size_t fragB = fragA + (size_t)KS * 2 * 32 * 4;      // [KS][2][32] float4
    static constexpr size_t tile = fragB + (size_t)KS * 2 * 32 * 4;       // [HP][132]
    static constexpr size_t das = tile + (size_t)HP * MID4_TP;            // [128][24] TF32 hi part of da
    static constexpr size_t das_lo = das + (size_t)MID4_R * MID4_DP;      // [128][24]
    static constexpr size_t b1 = das_lo + (size_t)MID4_R * MID4_DP;       // [HP]
    static constexpr size_t db1 = b1 + HP;                                // [8 warps][HP] per-warp column sums of dpre
    static constexpr size_t b2 = db1 + 8 * HP;                            // [16]
    static constexpr size_t total = b2 + 16;
};

__device__ __forceinline__ void mma_tf32(float (&d)[4], const float (&a)[4], float b0, float b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(__float_as_uint(a[0])), "r"(__float_as_uint(a[1])), "r"(__float_as_uint(a[2])), "r"(__float_as_uint(a[3])),
          "r"(__float_as_uint(b0)), "r"(__float_as_uint(b1)));
}

// tanh with ~1e-7 absolute error, 13 issue slots, branch-free: odd polynomial below 0.25 (truncation < 1e-8 relative),
// 1 - 2 / (1 + e^{2x}) above (ex2.approx / rcp.approx: absolute error ~2e-7 on a value >= 0.24).
__device__ __forceinline__ float tanh_fast(float x) {
    const float x2 = x * x;
    float p = 0.021869488536155203f;                 //  62/2835
    p = __fmaf_rn(p, x2, -0.053968253968253971f);    // -17/315
    p = __fmaf_rn(p, x2, 0.13333333333333333f);      //   2/15
    p = __fmaf_rn(p, x2, -0.33333333333333333f);     //  -1/3
    const float small = __fmaf_rn(x * x2, p, x);
    float e;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * 2.8853900817779268f));
    const float big = 1.f - __fdividef(2.f, 1.f + e);
    return fabsf(x) < 0.25f ? small : big;
}

// fast activations for the tensor-core variant (MUFU ex2 / rcp: absolute error ~1e-7)
__device__ __forceinline__ float act_fast(int act, float x) {
    if (act == ACT_TANH) return tanh_fast(x);
    if (act == ACT_RELU) return fmaxf(x, 0.f);
    float e;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * -1.4426950408889634f));
    return __fdividef(1.f, 1.f + e);
}

// hi = x rounded to TF32; lo = the exact remainder, NOT re-rounded: mma.sync reads only the TF32 bits of an operand
// register, i.e. truncates lo (relative error <= 2^-21 of x, sign uncorrelated with x) -- used for mma.sync operands only.
__device__ __forceinline__ void split_tf32_trunc_lo(float x, float& hi, float& lo) {
    hi = umma::rn_tf32(x);
    lo = x - hi;
}

template <int HP, bool FULL>      // FULL: B is a multiple of 128 (no row guards anywhere)
__global__ void __launch_bounds__(MID4_THREADS, 2)
bnn_mid4_kernel(const float* __restrict__ pre, const float* __restrict__ W, float* __restrict__ dW,
                const int32_t* __restrict__ y, BnnLayout L, float inv_S, double* __restrict__ loss,
                __half* __restrict__ dpT_hi, __half* __restrict__ dpT_lo, int64_t ldB, const float* __restrict__ scal) {
    using M = Mid4Smem<HP>;
    constexpr int KS = M::KS;
    extern __shared__ __align__(16) float sm[];
    float4* fragA = reinterpret_cast<float4*>(sm + M::fragA);
    float4* fragB = reinterpret_cast<float4*>(sm + M::fragB);
    float* tile = sm + M::tile;
    float* das_hi = sm + M::das;
    float* das_lo = sm + M::das_lo;
    float* b1s = sm + M::b1;
    float* db1s = sm + M::db1;
    float* b2s = sm + M::b2;
    __shared__ double red[32];

    const int H = L.H, C = L.C, B = L.B;
    const int s = blockIdx.y, b0 = blockIdx.x * MID4_R, tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    const float* Ws = W + (int64_t)s * L.ldw;
    float* dWs = dW + (int64_t)s * L.ldw;
    const float* W2 = Ws + L.oW2;

    // ---- phase A loads first (their latency overlaps the weight staging): pre[h][row] for this thread's 2 rows x 2*KS
    // hidden units.  Rows >= B and hidden units >= H are CLAMPED to valid addresses, not masked: invalid rows get da = 0
    // below, and hidden units >= H meet zero weights in both fragment sets and are never stored.
    const int r0 = 16 * warp + g, r1 = r0 + 8;                 // this thread's two rows inside the CTA block
    const bool ok0 = FULL || b0 + r0 < B, ok1 = FULL || b0 + r1 < B;
    float hA[KS][4];
    {
        const float* pc0 = pre + (int64_t)s * B * H + (ok0 ? b0 + r0 : B - 1);
        const float* pc1 = pre + (int64_t)s * B * H + (ok1 ? b0 + r1 : B - 1);
#pragma unroll
        for (int k = 0; k < KS; ++k) {
            const int h0 = min(8 * k + 2 * t, H - 1), h1 = min(8 * k + 2 * t + 1, H - 1);
            hA[k][0] = pc0[(int64_t)h0 * B];
            hA[k][1] = pc1[(int64_t)h0 * B];
            hA[k][2] = pc0[(int64_t)h1 * B];
            hA[k][3] = pc1[(int64_t)h1 * B];
        }
    }

    // ---- stage the per-sample layer-2 weights as ready-made (hi, lo) B fragments
    for (int idx = tid; idx < KS * 2 * 32; idx += MID4_THREADS) {
        const int ln = idx & 31, q = (idx >> 5) & 1, k = idx >> 6, gg = ln >> 2, tt = ln & 3;
        {   // phase A: B[k = hidden, n = class]: b0 = W2[8q + g][8k + 2t], b1 = W2[8q + g][8k + 2t + 1]
            const int c = 8 * q + gg, h0 = 8 * k + 2 * tt;
            const float w0 = (c < C && h0 < H) ? W2[(int64_t)c * H + h0] : 0.f;
            const float w1 = (c < C && h0 + 1 < H) ? W2[(int64_t)c * H + h0 + 1] : 0.f;
            float4 f;
            umma::split_tf32(w0, f.x, f.z);
            umma::split_tf32(w1, f.y, f.w);
            fragA[idx] = f;
        }
        {   // phase B: B[k = class, n = hidden]: b0 = W2[8q + 2t][8k + g], b1 = W2[8q + 2t + 1][8k + g]   (k = n-tile j)
            const int c0 = 8 * q + 2 * tt, h = 8 * k + gg;
            const float w0 = (c0 < C && h < H) ? W2[(int64_t)c0 * H + h] : 0.f;
            const float w1 = (c0 + 1 < C && h < H) ? W2[(int64_t)(c0 + 1) * H + h] : 0.f;
            float4 f;
            umma::split_tf32(w0, f.x, f.z);
            umma::split_tf32(w1, f.y, f.w);
            fragB[idx] = f;
        }
    }
    for (int idx = tid; idx < HP; idx += MID4_THREADS) b1s[idx] = idx < H ? Ws[L.ob1 + idx] : 0.f;
    if (tid < 16) b2s[tid] = tid < C ? Ws[L.ob2 + tid] : 0.f;
    __syncthreads();

    // ---- phase A: h = tanh(pre + b1) (kept in A-fragment registers and in the smem tile), a = h W2^T
    float ahh[2][4], acr[2][4];
#pragma unroll
    for (int q = 0; q < 2; ++q)
#pragma unroll
        for (int i = 0; i < 4; ++i) ahh[q][i] = acr[q][i] = 0.f;
    {
        float* tp = tile + (2 * t) * MID4_TP + r0;
#pragma unroll
        for (int k = 0; k < KS; ++k) {
            const float2 bb = *reinterpret_cast<const float2*>(b1s + 8 * k + 2 * t);
            float hi[4], lo[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float v = act_fast(L.act, hA[k][i] + (i < 2 ? bb.x : bb.y));
                hA[k][i] = v;
                split_tf32_trunc_lo(v, hi[i], lo[i]);
            }
            tp[k * 8 * MID4_TP] = hA[k][0];
            tp[k * 8 * MID4_TP + 8] = hA[k][1];
            tp[k * 8 * MID4_TP + MID4_TP] = hA[k][2];
            tp[k * 8 * MID4_TP + MID4_TP + 8] = hA[k][3];
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const float4 f = fragA[(k * 2 + q) * 32 + lane];
                mma_tf32(ahh[q], hi, f.x, f.y);
                mma_tf32(acr[q], lo, f.x, f.y);
                mma_tf32(acr[q], hi, f.z, f.w);
            }
        }
    }

    // ---- log-softmax over the classes: row r0 holds classes {2t, 2t+1, 8+2t, 9+2t} in a[q][0..1], row r1 in a[q][2..3]
    float dahi[2][4], dalo[2][4];            // phase-B A fragments: (r0, class 2t), (r1, 2t), (r0, 2t+1), (r1, 2t+1)
    float ll = 0.f;
    {
        const int lab0 = ok0 ? y[b0 + r0] : -1, lab1 = ok1 ? y[b0 + r1] : -1;
        float a[2][4];
        float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
        for (int q = 0; q < 2; ++q)
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int c = 8 * q + 2 * t + (i & 1);
                a[q][i] = c < C ? ahh[q][i] + acr[q][i] + b2s[c] : -INFINITY;
                if (i < 2) m0 = fmaxf(m0, a[q][i]);
                else m1 = fmaxf(m1, a[q][i]);
            }
        m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1)); m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 2));
        m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1)); m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 2));
        float ex[2][4];
        float se0 = 0.f, se1 = 0.f;
#pragma unroll
        for (int q = 0; q < 2; ++q)
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                ex[q][i] = expf(a[q][i] - (i < 2 ? m0 : m1));            // exp(-inf) = 0 for the pad classes
                if (i < 2) se0 += ex[q][i];
                else se1 += ex[q][i];
            }
        se0 += __shfl_xor_sync(0xffffffffu, se0, 1); se0 += __shfl_xor_sync(0xffffffffu, se0, 2);
        se1 += __shfl_xor_sync(0xffffffffu, se1, 1); se1 += __shfl_xor_sync(0xffffffffu, se1, 2);
        const float lse0 = m0 + logf(se0), lse1 = m1 + logf(se1);
        const float inv0 = 1.f / se0, inv1 = 1.f / se1;
        float da[2][4];
#pragma unroll
        for (int q = 0; q < 2; ++q)
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int c = 8 * q + 2 * t + (i & 1);
                const bool ok = (i < 2 ? ok0 : ok1) && c < C;
                const int lab = i < 2 ? lab0 : lab1;
                const float lse = i < 2 ? lse0 : lse1;
                const float sm_ = ex[q][i] * (i < 2 ? inv0 : inv1);
                da[q][i] = ok ? (c == lab ? 1.f : 0.f) - sm_ : 0.f;              // d ll / d a_c
                if (ok && c == lab) ll += a[q][i] - lse;
            }
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            split_tf32_trunc_lo(da[q][0], dahi[q][0], dalo[q][0]);
            split_tf32_trunc_lo(da[q][2], dahi[q][1], dalo[q][1]);
            split_tf32_trunc_lo(da[q][1], dahi[q][2], dalo[q][2]);
            split_tf32_trunc_lo(da[q][3], dahi[q][3], dalo[q][3]);
            *reinterpret_cast<float2*>(das_hi + r0 * MID4_DP + 8 * q + 2 * t) = make_float2(dahi[q][0], dahi[q][2]);
            *reinterpret_cast<float2*>(das_hi + r1 * MID4_DP + 8 * q + 2 * t) = make_float2(dahi[q][1], dahi[q][3]);
            *reinterpret_cast<float2*>(das_lo + r0 * MID4_DP + 8 * q + 2 * t) = make_float2(dalo[q][0], dalo[q][2]);
            *reinterpret_cast<float2*>(das_lo + r1 * MID4_DP + 8 * q + 2 * t) = make_float2(dalo[q][1], dalo[q][3]);
        }
    }

    // ---- phase B: dh = da W2, dpre = dh (1 - h^2) -> TF32 split, transposed store; db1 column sums
    {
        // output pointers walk down the hidden axis: element (h0 = 2t [+1], row r0 [+8]) of this sample's block
        __half* ohi0 = dpT_hi + ((int64_t)s * HP + 2 * t) * ldB + b0 + r0;
        __half* olo0 = dpT_lo + ((int64_t)s * HP + 2 * t) * ldB + b0 + r0;
        __half* ohi1 = ohi0 + ldB;
        __half* olo1 = olo0 + ldB;
        const float sD = dpre_scale(scal);
        const int64_t step = 8 * ldB;
#pragma unroll
        for (int j = 0; j < KS; ++j) {
            float dhh[4] = {0.f, 0.f, 0.f, 0.f}, dcr[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const float4 f = fragB[(j * 2 + q) * 32 + lane];
                mma_tf32(dhh, dahi[q], f.x, f.y);
                mma_tf32(dcr, dalo[q], f.x, f.y);
                mma_tf32(dcr, dahi[q], f.z, f.w);
            }
            // C fragment: (r0, h0), (r0, h0+1), (r1, h0), (r1, h0+1) with h0 = 8j + 2t  <->  hA[j][0], [2], [1], [3]
            const int h0 = 8 * j + 2 * t;
            float dp[4];
            dp[0] = (dhh[0] + dcr[0]) * act_grad_from_h(L.act, hA[j][0]);
            dp[1] = (dhh[1] + dcr[1]) * act_grad_from_h(L.act, hA[j][2]);
            dp[2] = (dhh[2] + dcr[2]) * act_grad_from_h(L.act, hA[j][1]);
            dp[3] = (dhh[3] + dcr[3]) * act_grad_from_h(L.act, hA[j][3]);
            __half hi[4], lo[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) split_f16(dp[i] * sD, hi[i], lo[i]);
            // hidden units >= H: dp == 0 there (zero fragB weights) and the pad rows of dpT exist -> no guard needed
            if (ok0) { ohi0[0] = hi[0]; olo0[0] = lo[0]; ohi1[0] = hi[1]; olo1[0] = lo[1]; }
            if (ok1) { ohi0[8] = hi[2]; olo0[8] = lo[2]; ohi1[8] = hi[3]; olo1[8] = lo[3]; }
            ohi0 += step; olo0 += step; ohi1 += step; olo1 += step;
            float c0 = dp[0] + dp[2], c1 = dp[1] + dp[3];        // column sums over this warp's 16 rows
#pragma unroll
            for (int o = 4; o < 32; o <<= 1) {
                c0 += __shfl_xor_sync(0xffffffffu, c0, o);
                c1 += __shfl_xor_sync(0xffffffffu, c1, o);
            }
            if (g == 0) *reinterpret_cast<float2*>(db1s + warp * HP + h0) = make_float2(c0, c1);   // per-warp partial
        }
    }
    __syncthreads();

    // ---- phase C: dW2[c, h] = sum_b da[b, c] h[b, h] over the CTA's 128 rows; warp w owns hidden n-tiles w and w + 8
    auto phase_c = [&](auto ntag) {
        constexpr int NT = decltype(ntag)::value;
        float chh[NT][4], ccr[NT][4];
#pragma unroll
        for (int q = 0; q < NT; ++q)
#pragma unroll
            for (int i = 0; i < 4; ++i) chh[q][i] = ccr[q][i] = 0.f;
        const float* dh_ = das_hi + t * MID4_DP + g;
        const float* dl_ = das_lo + t * MID4_DP + g;
        const float* tb = tile + (8 * warp + g) * MID4_TP + t;
#pragma unroll 4
        for (int kb = 0; kb < MID4_R / 8; ++kb) {
            // A = da^T: (class g, row 8kb+t), (class g+8, row 8kb+t), (class g, row 8kb+t+4), (class g+8, row 8kb+t+4)
            float ahi[4], alo[4];
            ahi[0] = dh_[kb * 8 * MID4_DP];
            ahi[1] = dh_[kb * 8 * MID4_DP + 8];
            ahi[2] = dh_[(kb * 8 + 4) * MID4_DP];
            ahi[3] = dh_[(kb * 8 + 4) * MID4_DP + 8];
            alo[0] = dl_[kb * 8 * MID4_DP];
            alo[1] = dl_[kb * 8 * MID4_DP + 8];
            alo[2] = dl_[(kb * 8 + 4) * MID4_DP];
            alo[3] = dl_[(kb * 8 + 4) * MID4_DP + 8];
#pragma unroll
            for (int q = 0; q < NT; ++q) {
                float bh0, bl0, bh1, bl1;
                split_tf32_trunc_lo(tb[q * 64 * MID4_TP + kb * 8], bh0, bl0);          // B = h: (row 8kb+t, hidden 8j+g)
                split_tf32_trunc_lo(tb[q * 64 * MID4_TP + kb * 8 + 4], bh1, bl1);
                mma_tf32(chh[q], ahi, bh0, bh1);
                mma_tf32(ccr[q], alo, bh0, bh1);
                mma_tf32(ccr[q], ahi, bl0, bl1);
            }
        }
#pragma unroll
        for (int q = 0; q < NT; ++q) {
            const int h0 = 8 * (warp + 8 * q) + 2 * t;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int c = g + (i >= 2 ? 8 : 0), h = h0 + (i & 1);
                if (c < C && h < H) atomicAdd(&dWs[L.oW2 + (int64_t)c * H + h], chh[q][i] + ccr[q][i]);
            }
        }
    };
    if (warp + 8 < KS) phase_c(std::integral_constant<int, 2>());
    else if (warp < KS) phase_c(std::integral_constant<int, 1>());
    if (warp == 7 && lane < C) {
        float acc = 0.f;
        for (int rr = 0; rr < MID4_R; ++rr) acc += das_hi[rr * MID4_DP + lane] + das_lo[rr * MID4_DP + lane];
        atomicAdd(&dWs[L.ob2 + lane], acc);
    }
    for (int idx = tid; idx < H; idx += MID4_THREADS) {
        float acc = 0.f;
#pragma unroll
        for (int w = 0; w < MID4_THREADS / 32; ++w) acc += db1s[w * HP + idx];
        atomicAdd(&dWs[L.ob1 + idx], acc);
    }
    double tot = block_sum<double>((double)ll, red);
    if (tid == 0) atomicAdd(loss, -tot * (double)inv_S);
}

template <int HP>
static int launch_mid4(const float* pre, const float* W, float* dW, const int32_t* y, const BnnLayout& L, int S, float inv_S,
                       double* loss, __half* dph, __half* dpl, int64_t ldB, const float* scal, cudaStream_t stream) {
    const size_t smem = Mid4Smem<HP>::total * sizeof(float);
    dim3 grid((L.B + MID4_R - 1) / MID4_R, S);
    if (L.B % MID4_R == 0) {
        BRN_CUDA_OK(cudaFuncSetAttribute(bnn_mid4_kernel<HP, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        bnn_mid4_kernel<HP, true><<<grid, MID4_THREADS, smem, stream>>>(pre, W, dW, y, L, inv_S, loss, dph, dpl, ldB, scal);
    } else {
        BRN_CUDA_OK(cudaFuncSetAttribute(bnn_mid4_kernel<HP, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        bnn_mid4_kernel<HP, false><<<grid, MID4_THREADS, smem, stream>>>(pre, W, dW, y, L, inv_S, loss, dph, dpl, ldB, scal);
    }
    BRN_LAUNCH_OK("bnn_mid4_kernel");
    return 0;
}

// ---------------------------------------------------------------------------------------------------
// layer-1 sampler: noise + W1_s = mu + softplus(rho) eps_s + fp16 (hi, lo) split, scaled by w1_scale, in the padded K-major
// layout Wh/Wl [(s * Hp + h)][ldP] the GEMMs read through TMA.  Sample-group version (P % 4 == 0): one thread = 4
// consecutive weights, walking SG consecutive samples; sigma is evaluated once per thread.
// Pad rows h in [H, Hp) are never written: they only feed accumulator columns the epilogues mask.
// ---------------------------------------------------------------------------------------------------
template <int SG>
__global__ void __launch_bounds__(256)
sample_w1_group_kernel(const float* __restrict__ mu, const float* __restrict__ rho, const float* __restrict__ eps_in,
                       int64_t lde_in, float* __restrict__ eps_out, int64_t lde_out, __half* __restrict__ hi,
                       __half* __restrict__ lo, int H, int P, int Hp, int64_t ldP, brn_sample_range r, uint32_t var_id,
                       const float* __restrict__ scal) {
    const int64_t qq = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (qq * 4 >= (int64_t)H * P) return;
    const int h = (int)((qq * 4) / P), p = (int)((qq * 4) - (int64_t)h * P);
    const int64_t i = (int64_t)h * P + p;
    const float sc = w1_scale(scal);
    const float4 m = *reinterpret_cast<const float4*>(mu + i);
    const float4 rh = *reinterpret_cast<const float4*>(rho + i);
    const float4 sg = make_float4(softplusf(rh.x), softplusf(rh.y), softplusf(rh.z), softplusf(rh.w));
    const int s_begin = blockIdx.y * SG, s_end = min(r.s_local, s_begin + SG);
    const int64_t o0 = (int64_t)h * ldP + p;
#pragma unroll 2
    for (int s = s_begin; s < s_end; ++s) {
        float4 e;
        if (eps_in) {
            e = *reinterpret_cast<const float4*>(eps_in + (int64_t)s * lde_in + i);
        } else {
            Normal4 n = philox_normal4(r.seed, philox_offset(r), var_id, (uint32_t)(r.s0 + s), (uint32_t)(i >> 2));
            e = make_float4(n.v[0], n.v[1], n.v[2], n.v[3]);
        }
        *reinterpret_cast<float4*>(eps_out + (int64_t)s * lde_out + i) = e;
        __half vh[4], vl[4];
        split_f16(__fmaf_rn(sg.x, e.x, m.x) * sc, vh[0], vl[0]);
        split_f16(__fmaf_rn(sg.y, e.y, m.y) * sc, vh[1], vl[1]);
        split_f16(__fmaf_rn(sg.z, e.z, m.z) * sc, vh[2], vl[2]);
        split_f16(__fmaf_rn(sg.w, e.w, m.w) * sc, vh[3], vl[3]);
        const int64_t o = (int64_t)s * Hp * ldP + o0;
        uint2 ph, pl;
        ph.x = (uint32_t)__half_as_ushort(vh[0]) | ((uint32_t)__half_as_ushort(vh[1]) << 16);
        ph.y = (uint32_t)__half_as_ushort(vh[2]) | ((uint32_t)__half_as_ushort(vh[3]) << 16);
        pl.x = (uint32_t)__half_as_ushort(vl[0]) | ((uint32_t)__half_as_ushort(vl[1]) << 16);
        pl.y = (uint32_t)__half_as_ushort(vl[2]) | ((uint32_t)__half_as_ushort(vl[3]) << 16);
        *reinterpret_cast<uint2*>(hi + o) = ph;
        *reinterpret_cast<uint2*>(lo + o) = pl;
    }
}

// any shape / alignment: one thread per (p, h, s), noise already materialised in eps [S][lde]
__global__ void sample_w1_generic_kernel(const float* __restrict__ mu, const float* __restrict__ rho, const float* __restrict__ eps,
                                         int64_t lde, __half* __restrict__ hi, __half* __restrict__ lo, int H, int P, int Hp,
                                         int64_t ldP, const float* __restrict__ scal) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x, h = blockIdx.y, s = blockIdx.z;
    if (p >= P) return;
    const int64_t i = (int64_t)h * P + p;
    __half vh, vl;
    split_f16(__fmaf_rn(softplusf(rho[i]), eps[(int64_t)s * lde + i], mu[i]) * w1_scale(scal), vh, vl);
    const int64_t o = ((int64_t)s * Hp + h) * ldP + p;
    hi[o] = vh;
    lo[o] = vl;
}

constexpr int BNN_UMMA_HP = 104;     // padded hidden width of the instantiated tcgen05 variant (multiple of 8)
constexpr int BNN_UMMA_BK = 16;      // K chunk: 16 words = 64 bytes = 32 fp16 (64-byte swizzle), 5-stage TMA ring
constexpr int BNN_UMMA_NSAMP = 2;    // samples per MMA N tile (N = 208)

// workspace of the tcgen05 variant (appended to the SIMT variant's blocks by BnnWorkspace in bnn.cu)
struct BnnTcWorkspace {
    __half *Xh, *Xl, *Xth, *Xtl, *Wh, *Wl, *dph, *dpl;   // fp16 (hi, lo) operands
    float* scal;                                         // operand bounds (SC_*), zeroed per call
    int64_t ldP, ldB;
    template <class Take>
    void carve(Take&& take, const BnnLayout& L, int S) {
        ldP = (L.P + 7) / 8 * 8;
        ldB = (L.B + 7) / 8 * 8;
        auto half_block = [&](size_t n) { return reinterpret_cast<__half*>(take((n + 1) / 2)); };
        Xh = half_block((size_t)L.B * ldP); Xl = half_block((size_t)L.B * ldP);
        Xth = half_block((size_t)L.P * ldB); Xtl = half_block((size_t)L.P * ldB);
        const size_t rowsW = (size_t)(S + BNN_UMMA_NSAMP) * BNN_UMMA_HP;
        Wh = half_block(rowsW * ldP); Wl = half_block(rowsW * ldP);
        dph = half_block(rowsW * ldB); dpl = half_block(rowsW * ldB);
        scal = take(SC_SLOTS);
    }
};

// Layer-1 pieces of the tcgen05 variant, shared by the two-layer evaluation below and the deep networks (bnn_deep.cuh).
// Sampling-stage part for W1 (vars w1): operand bounds (scal[SC_W2] from w2), noise + W1_s split into the forward GEMM's
// fp16 pairs, finite padding of the odd tail sample block.
static int bnn_tc_sample_w1(const brn_mf_var& w1, const brn_mf_var& w2, int H, int P, int64_t ldw, const brn_sample_range* r,
                            const BnnTcWorkspace& ws, float* ws_eps, cudaStream_t stream) {
    constexpr int HP = BNN_UMMA_HP, NS = BNN_UMMA_NSAMP;
    const int S = r->s_local;
    const int64_t n1 = (int64_t)H * P, n2 = w2.numel;
    BRN_CUDA_OK(cudaMemsetAsync(ws.scal, 0, sizeof(float) * SC_SLOTS, stream));
    // operand bounds (device scalars): injected noise is not bounded a priori
    if (w1.eps) if (int e = launch_absmax(w1.eps, (int64_t)S * n1, ws.scal + SC_EPS, stream)) return e;
    if (w2.eps) if (int e = launch_absmax(w2.eps, (int64_t)S * n2, ws.scal + SC_EPS, stream)) return e;
    bnn_bounds_kernel<<<(unsigned)std::min<int64_t>((n1 + n2 + 255) / 256, 296), 256, 0, stream>>>(
        w1.mu, w1.rho, n1, w2.mu, w2.rho, n2, ws.scal);
    BRN_LAUNCH_OK("bnn_bounds_kernel");
    const bool fast = (P % 4 == 0) && ((uintptr_t)w1.mu % 16 == 0) && ((uintptr_t)w1.rho % 16 == 0) &&
                      (!w1.eps || ((uintptr_t)w1.eps % 16 == 0));
    if (fast) {
        constexpr int SG = 8;
        dim3 grid((unsigned)((n1 / 4 + 255) / 256), (unsigned)((S + SG - 1) / SG));
        sample_w1_group_kernel<SG><<<grid, 256, 0, stream>>>(w1.mu, w1.rho, w1.eps, n1, ws_eps, ldw, ws.Wh, ws.Wl, H, P, HP, ws.ldP,
                                                             *r, w1.var_id, ws.scal);
        BRN_LAUNCH_OK("sample_w1_group_kernel");
    } else {
        if (w1.eps)
            BRN_CUDA_OK(cudaMemcpy2DAsync(ws_eps, ldw * sizeof(float), w1.eps, n1 * sizeof(float), n1 * sizeof(float), S,
                                          cudaMemcpyDeviceToDevice, stream));
        else if (int e = launch_philox_fill(ws_eps, ldw, n1, w1.var_id, *r, stream)) return e;
        dim3 grid((P + 255) / 256, H, S);
        sample_w1_generic_kernel<<<grid, 256, 0, stream>>>(w1.mu, w1.rho, ws_eps, ldw, ws.Wh, ws.Wl, H, P, HP, ws.ldP, ws.scal);
        BRN_LAUNCH_OK("sample_w1_generic_kernel");
    }
    if (S % NS) {   // the odd tail tile reads one more sample block: keep it finite
        BRN_CUDA_OK(cudaMemsetAsync(ws.Wh + (size_t)S * HP * ws.ldP, 0, sizeof(__half) * HP * ws.ldP, stream));
        BRN_CUDA_OK(cudaMemsetAsync(ws.Wl + (size_t)S * HP * ws.ldP, 0, sizeof(__half) * HP * ws.ldP, stream));
        BRN_CUDA_OK(cudaMemsetAsync(ws.dph + (size_t)S * HP * ws.ldB, 0, sizeof(__half) * HP * ws.ldB, stream));
        BRN_CUDA_OK(cudaMemsetAsync(ws.dpl + (size_t)S * HP * ws.ldB, 0, sizeof(__half) * HP * ws.ldB, stream));
    }
    return 0;
}

// first read of the minibatch: X's bound and its fp16 pairs (row-major for the forward GEMM, transposed for the backward)
static int bnn_tc_split_x(const float* X, int B, int P, const BnnTcWorkspace& ws, cudaStream_t stream) {
    if (int e = wait_data_ready(stream)) return e;
    if (int e = launch_absmax(X, (int64_t)B * P, ws.scal + SC_X, stream)) return e;
    dim3 grid((B + 31) / 32, (P + 31) / 32), block(32, 8);
    split_f16_kernel<<<grid, block, 0, stream>>>(X, P, B, P, ws.Xh, ws.Xl, ws.ldP, ws.Xth, ws.Xtl, ws.ldB, ws.scal);
    BRN_LAUNCH_OK("split_f16_kernel");
    return 0;
}

// TMEM accumulation chain = 2 x 32 words = 128 fp16 elements of K between register drains (umma_gemm.cuh): the error
// of the evaluation grows with the chain (max gradient error / scale at the C3 shape: 0.9e-6 / 1.1e-6 / 1.3e-6 /
// 2.3e-6 for 1 / 2 / 4 / 8, profiles/tools/bnn_err_probe.py) -- 128 elements is the chain length round 1 settled on.
// The backward GEMM's accumulator is the per-sample weight gradient, summed over 256 samples afterwards: its chain
// may be twice as long (measured: no change of the parity margins, 8 us per evaluation).
constexpr int BNN_UMMA_DRAIN = 2, BNN_UMMA_DRAIN_BWD = 4;

// pre_s^T [S][H][B] = (X . W1_s^T)^T, coalesced across the warp's rows b
static int bnn_tc_gemm_fwd(int B, int P, int H, int S, const BnnTcWorkspace& ws, float* ws_pre, cudaStream_t stream) {
    constexpr int BN = BNN_UMMA_HP * BNN_UMMA_NSAMP;
    EpiStore::Params ep;
    ep.out = ws_pre; ep.rows = B; ep.row_stride = 1; ep.col_stride = B; ep.blk_stride = (int64_t)B * H;
    ep.blk_valid = H; ep.col_limit = 0; ep.total_blks = S;
    ep.bound_a = ws.scal + SC_X; ep.bound_b = ws.scal + SC_W1; ep.bound_b_mult = 1.f;
    return launch_umma_nt_kind<BN, BNN_UMMA_BK, EpiStore, 8, 0, 4, 1>(ws.Xh, ws.Xl, B, ws.ldP, ws.Wh, ws.Wl, S * BNN_UMMA_HP, ws.ldP, P, 0,
                                                                        BNN_UMMA_DRAIN, ep, stream);
}

// dW1_s[h][p] = D[p, (s, h)] = (dpre_s^T X)[h][p] from the fp16 pairs ws.dph / ws.dpl, which were scaled by
// p2_scale(dpre_mult * *dpre_bound)
static int bnn_tc_gemm_bwd(int B, int P, int H, int S, int64_t ldw, const BnnTcWorkspace& ws, float* ws_dW1, const float* dpre_bound,
                           float dpre_mult, cudaStream_t stream) {
    constexpr int NS = BNN_UMMA_NSAMP, BN = BNN_UMMA_HP * NS;
    // K-split tail (see UnitIter): the dW1 blocks of the samples in the split n-tiles take atomic partial sums
    const int sms = device_sm_count();
    const UmmaSplitPlan plan = umma_plan<BN, 2 * BNN_UMMA_BK>(P, S * BNN_UMMA_HP, B, sms, true);
    if (plan.first_split_ntile >= 0) {
        const int s_first = plan.first_split_ntile * NS;
        if (s_first < S)
            BRN_CUDA_OK(cudaMemset2DAsync(ws_dW1 + (size_t)s_first * ldw, ldw * sizeof(float), 0, (size_t)H * P * sizeof(float),
                                          S - s_first, stream));
    }
    EpiStore::Params ep;
    ep.out = ws_dW1; ep.rows = P; ep.row_stride = 1; ep.col_stride = P; ep.blk_stride = ldw;
    ep.blk_valid = H; ep.col_limit = 0; ep.total_blks = S;
    ep.bound_a = ws.scal + SC_X; ep.bound_b = dpre_bound; ep.bound_b_mult = dpre_mult;
    return launch_umma_nt_kind<BN, BNN_UMMA_BK, EpiStore, 8, 0, 4, 1>(ws.Xth, ws.Xtl, P, ws.ldB, ws.dph, ws.dpl, S * BNN_UMMA_HP, ws.ldB, B,
                                                                        0, BNN_UMMA_DRAIN_BWD, ep, stream, true);
}

// The tcgen05 variant of brn_bnn_elbo_fwd_bwd: sampler -> forward GEMM -> mid kernel -> backward GEMM -> statistics.
// forward_only (brn_bnn_predict) stops after the forward GEMM.
static int bnn_tc_eval(const float* X, const int32_t* y, const BnnLayout& L, const brn_mf_var vars[4], const brn_sample_range* r,
                       const BnnTcWorkspace& ws, float* ws_eps, float* ws_W, float* ws_dW, float* ws_pre, float* ws_stats,
                       int with_prior, double* loss, cudaStream_t stream, bool forward_only = false) {
    const int B = L.B, P = L.P, H = L.H, S = r->s_local;
    const int64_t offs[4] = {L.oW1, L.ob1, L.oW2, L.ob2};
    const float inv_S = 1.0f / (float)r->s_total;
    {
        StageTimer st("bnn.sample_weights", stream);
        if (int e = bnn_tc_sample_w1(vars[0], vars[2], H, P, L.ldw, r, ws, ws_eps + offs[0], stream)) return e;
        // small variables: noise, sampled values, and zeroed per-sample gradient slots (accumulated into by the mid stage)
        if (int e = launch_sample_multi(vars + 1, offs + 1, 3, ws_eps, ws_W, L.ldw, *r, stream, ws_dW)) return e;
        // first read of the minibatch: everything above overlaps a host->device copy announced by brn_set_data_ready_event
        if (int e = bnn_tc_split_x(X, B, P, ws, stream)) return e;
    }
    {
        StageTimer st("bnn.gemm_fwd", stream);
        if (int e = bnn_tc_gemm_fwd(B, P, H, S, ws, ws_pre, stream)) return e;
    }
    if (forward_only) return 0;          // brn_bnn_predict: pre^T [S][H][B] is all it needs
    {
        StageTimer st("bnn.mid", stream);
        if (int e = launch_mid4<BNN_UMMA_HP>(ws_pre, ws_W, ws_dW, y, L, S, inv_S, loss, ws.dph, ws.dpl, ws.ldB, ws.scal, stream)) return e;
    }
    {
        StageTimer st("bnn.gemm_bwd", stream);
        // dpre = (W2^T da) act'(h) with sum_c |da_c| <= 2 and |act'| <= 1:  |dpre| <= 2 scal[SC_W2]
        if (int e = bnn_tc_gemm_bwd(B, P, H, S, L.ldw, ws, ws_dW + L.oW1, ws.scal + SC_W2, 2.f, stream)) return e;
    }
    StageTimer st5("bnn.reduce_finalize", stream);
    return launch_mf_reduce_finalize_multi(vars, offs, 4, L.numel, ws_eps, L.ldw, ws_dW, L.ldw, ws_stats, *r, with_prior, loss, stream, 0);
}

}  // namespace brn
