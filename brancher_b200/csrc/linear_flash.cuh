// K2 / K4a "flash" kernel: Bernoulli log-likelihood and its weight gradient for S weight vectors in ONE pass over X, with
// both contractions on tcgen05 and the intermediate d = y - sigmoid(logit) never leaving the SM.
//
//   per 64-row block of X (CTA = one tile of 128 weight vectors x a strided set of row blocks):
//     MMA1   L[s, r]   = sum_f W[s, f] X[r, f]              M = 128 vectors, N = 64 rows,  K = F   (D1 in TMEM, 64 columns)
//     epilogue         d = y_r - sigmoid(L), ll += y L - softplus(L); d -> fp16 (hi, lo) pair, written with tcgen05.st to
//                      TENSOR memory as the A operand of MMA2 (the thread that owns TMEM lane s writes row s: no
//                      transposition; DTMEM = 0 keeps the round-trip through a K-major shared-memory tile)
//     MMA2   dW[s, f] += sum_r d[s, r] X[r, f]             M = 128 vectors, N = F,        K = 64 rows (D2 in TMEM, F columns)
//   The SAME shared-memory image of the X block serves MMA1 as a K-major B operand (K = f, contiguous) and MMA2 as an
//   MN-major B operand (N = f contiguous, K = rows): no transposed copy of X exists anywhere.
//
// Replaces the staged pair (logits GEMM -> d^T through HBM -> gradient GEMM): at C2 that pair moved 4 GB of d^T out and
// back per evaluation and read X twice (row-major and a per-chunk transposed copy).  Operands are fp16 (hi, lo) pairs
// ("3xFP16", see bnn_tc.cuh), scaled by powers of two: X and W are split once per call by small streaming kernels (X: one
// read + one write of its own size, or once per data matrix: brn_linear_prepare_x) and arrive by TMA in the swizzled UMMA
// layout, five blocks in flight per SM, the block's targets y riding along (bulk copy); d is in (-1, 1) and scaled by 2^13.  (A first version converted fp32 X inside the kernel from a 32 KB staging area: with only that
// much in flight per SM the X feed was latency-bound at ~5000 cycles per block against 1536 of tensor work.)
// Accuracy: D2's accumulation chain is 128 rows long (two blocks) between round-to-nearest drains into registers.
// Warp roles (20 warps): 0 = TMA producer, 1 = logits-MMA issuer, 2 = gradient-MMA issuer, 3 idle, 4-19 = epilogue in two
// groups of 8 that take the blocks alternately.  TMEM: D1 3 x 64 columns, d 64, D2 2 x 128.  History: profiles/r2f_flash_history.txt.
#pragma once
#include <cuda_fp16.h>
#include "umma_gemm.cuh"
#include <algorithm>
#include <stdlib.h>
#include <type_traits>

namespace brn {

constexpr int LF_ROWS = 64;            // rows of X per block (N of MMA1, K of MMA2)
constexpr int LF_MT = 128;             // weight vectors per CTA tile (M of both MMAs)
constexpr int LF_FMAX = 128;           // features (K of MMA1, N of MMA2): multiple of 16, at most 128
constexpr int LF_XSTAGES_SMEM_D = 4;   // X blocks (fp16 pair images, 32 KB each) in flight; 5 when the d tile lives in TMEM
constexpr int LF_D1BUF = 3;            // logits accumulators in TMEM: the logits MMA runs two blocks ahead of the gradient MMA
constexpr int LF_THREADS = 640;        // 20 warps: TMA, 2 MMA issuers, 1 idle | 16 epilogue
constexpr int LF_EPI_WARP0 = 4, LF_EPI_WARPS = 16;
constexpr int LF_EROWS = 32;           // rows of a block per epilogue warp (two warps of one group cover a block)
constexpr int LF_EFEAT = 32;           // gradient features per epilogue warp (all 16 warps drain every chain)
constexpr int LF_D2_CHAIN = 2;         // blocks per D2 accumulation chain
constexpr float LF_D_SCALE = 8192.f;   // 2^13: |d| < 1

template <int DTMEM>
struct LinearFlashSmem {
    static constexpr int XSTAGES = DTMEM ? LF_XSTAGES_SMEM_D + 1 : LF_XSTAGES_SMEM_D;
    static constexpr int W_BYTES = 2 * LF_MT * LF_FMAX * 2;                 // (hi, lo) [128][128] fp16 = 64 KB
    static constexpr int X16_BYTES = 2 * LF_ROWS * LF_FMAX * 2;             // (hi, lo) [64][128] fp16 = 32 KB
    static constexpr int D_BYTES = DTMEM ? 0 : 2 * LF_MT * LF_ROWS * 2;     // (hi, lo) [128][64] fp16 = 32 KB (shared-memory d tile)
    static constexpr int off_w = 0;
    static constexpr int off_x16 = off_w + W_BYTES;
    static constexpr int off_d = off_x16 + XSTAGES * X16_BYTES;
    static constexpr int off_y = off_d + D_BYTES;                           // y of the block in each X stage: 64 floats
    static constexpr int Y_BYTES = LF_ROWS * 4;
    static constexpr int TOTAL = off_y + XSTAGES * Y_BYTES + 1024;          // + alignment slack
    static_assert(TOTAL <= 227 * 1024, "shared memory budget exceeded");
};

// kind::f16, fp16 operands, fp32 accumulate; b_mn: B operand is MN-major
__host__ __device__ constexpr uint32_t idesc_f16_major(int M, int N, bool b_mn) {
    return (1u << 4) | ((b_mn ? 1u : 0u) << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void bulk_copy_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(umma::smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(umma::smem_u32(bar))
                 : "memory");
}

// packed fp32 pairs (one issue slot for two lanes of work; sm_100)
__device__ __forceinline__ uint64_t f2_pack(float lo, float hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void f2_unpack(uint64_t v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ uint64_t f2_mul(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ uint64_t f2_add(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ uint64_t f2_fma(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}

struct LinearFlashParams {
    const float* y; int64_t N; int F; int S;
    const float* scal_w; const float* scal_x;      // max |W|, max |X|  (device scalars)
    float* part;                  // [groups][S_pad][F] partial gradients (+ d ll / d W), one slice per row group
    int64_t part_stride;          // S_pad * F
    double* loss; float loss_scale;
    int groups;
    int y_bulk;                   // y is 16-byte aligned: full blocks of it travel with the X block (bulk copy) into shared memory
    const float* scal_y;          // Gaussian: max |y|  (device scalar)
    double* R;                    // Gaussian: [S] += sum of squared residuals per vector (loss and loss_scale unused)
                                  // Cauchy: [S] += sum log1p(z^2);  Laplace: [S] += sum |r|
    const float* sigma;           // Cauchy: [S] noise scale per vector
    double* T;                    // Cauchy: [S] += sum z^2 / (1 + z^2)
};

// tcgen05.mma kind::f16 with both shared-memory descriptors given as (low word, shared high word)
__device__ __forceinline__ void mma_f16_lohi(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t hi, uint32_t idesc, bool accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
        "setp.ne.b32 p, %5, 0;\n\t"
        "mov.b64 da, {%1, %3};\n\t"
        "mov.b64 db, {%2, %3};\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, p;\n\t}"
        ::"r"(d_tmem), "r"(a_lo), "r"(b_lo), "r"(hi), "r"(idesc), "r"((uint32_t)accumulate)
        : "memory");
}

// tcgen05.mma kind::f16 with the A operand in TENSOR MEMORY (lane = row of A, one 32-bit column = two consecutive K elements)
__device__ __forceinline__ void mma_f16_ts_lohi(uint32_t d_tmem, uint32_t a_tmem, uint32_t b_lo, uint32_t hi, uint32_t idesc, bool accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 db;\n\t"
        "setp.ne.b32 p, %5, 0;\n\t"
        "mov.b64 db, {%2, %3};\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %4, p;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "r"(b_lo), "r"(hi), "r"(idesc), "r"((uint32_t)accumulate)
        : "memory");
}
// registers -> TMEM: thread i of the warp writes lane (lane_base + i), 16 consecutive 32-bit columns
__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t (&v)[16]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
                 ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
                   "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
                 : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// KS1 = F / 16 at compile time (the logits MMA loop is then fully unrolled), 0 = any F.
// DTMEM: the d tile (A operand of the gradient MMA) lives in tensor memory (64 columns: hi pair words, lo pair words) instead of
// shared memory -- the epilogue thread that owns TMEM lane s writes row s with tcgen05.st: no shared-memory round trip, no
// generic -> async proxy fence, half the shared-memory operand reads of the gradient MMA.
// LIK: 0 = Bernoulli (d = y - sigmoid(l), loss += loss_scale * sum ll), 1 = Gaussian residuals (d = r = y - l, R[s] += sum r^2;
// the noise scale is applied afterwards, per vector, by the caller), 2 = Cauchy (z = r / sigma_s, d = z / (1 + z^2),
// R[s] += sum log1p(z^2), T[s] += sum z^2 / (1 + z^2)), 3 = Laplace (d = sign(r), R[s] += sum |r|; sigma applied afterwards).
template <int KS1, int DTMEM, int LIK = 0>
__global__ void __launch_bounds__(LF_THREADS, 1)
linear_flash_kernel(const __grid_constant__ CUtensorMap tmWh, const __grid_constant__ CUtensorMap tmWl,
                    const __grid_constant__ CUtensorMap tmXh, const __grid_constant__ CUtensorMap tmXl, LinearFlashParams p) {
    using SM = LinearFlashSmem<DTMEM>;
    constexpr int LF_XSTAGES = SM::XSTAGES;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    __shared__ __align__(8) uint64_t w_full, x_full[LF_XSTAGES], x_empty[LF_XSTAGES], d1_full[LF_D1BUF], d1_empty[LF_D1BUF],
        d_full[2], d_empty[2], acc2_full[2], acc2_empty[2];
    __shared__ uint32_t tmem_base_slot;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int st = blockIdx.x, g = blockIdx.y;                      // vector tile, row group
    const int F = p.F, FB = (F + 63) / 64;                          // 64-feature boxes
    const int64_t n_blocks = (p.N + LF_ROWS - 1) / LF_ROWS;
    const int my_blocks = g < n_blocks ? (int)((n_blocks - g + p.groups - 1) / p.groups) : 0;     // N < 2^31: fits an int

    if (threadIdx.x == 0) {
        umma::tma_prefetch_desc(&tmWh); umma::tma_prefetch_desc(&tmWl);
        umma::tma_prefetch_desc(&tmXh); umma::tma_prefetch_desc(&tmXl);
        umma::mbar_init(&w_full, 1);
        for (int s = 0; s < LF_XSTAGES; ++s) { umma::mbar_init(&x_full[s], 1); umma::mbar_init(&x_empty[s], 1); }
        for (int b = 0; b < LF_D1BUF; ++b) { umma::mbar_init(&d1_full[b], 1); umma::mbar_init(&d1_empty[b], LF_EPI_WARPS / 2); }
        for (int b = 0; b < 2; ++b) { umma::mbar_init(&acc2_full[b], 1); umma::mbar_init(&acc2_empty[b], LF_EPI_WARPS); }
        // the ONE d tile is handed over through barriers indexed by block parity (= epilogue group): with a single barrier
        // a group running two phases behind would alias on the phase parity now that the two MMA threads are not ordered
        for (int b = 0; b < 2; ++b) { umma::mbar_init(&d_full[b], LF_EPI_WARPS / 2); umma::mbar_init(&d_empty[b], 1); }
        umma::fence_barrier_init();
    }
    if (warp == 1) umma::tmem_alloc(&tmem_base_slot, 512);
    umma::tc_fence_before();
    __syncthreads();
    umma::tc_fence_after();
    const uint32_t tmem_base = tmem_base_slot;
    const uint32_t t_d1 = tmem_base, t_d2 = tmem_base + 256;        // D1: 3 x 64 columns at 0 / 64 / 128; D2: 2 x 128 at 256 / 384
    const uint32_t t_dt = tmem_base + 192;                          // d tile (DTMEM): hi words at 192..223, lo words at 224..255

    // register budget: the CTA owns 96 registers x 640 threads (launch bounds); setmaxnreg only moves registers INSIDE that
    // allocation (asking for more blocks forever), so per warpgroup 32 + 4 x 112 = 480 = 5 x 96
    if (warp < LF_EPI_WARP0) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 32;");
    if (warp == 0) {
        // ===================== producer: W tile once, then the X blocks (rows past N are zero-filled by TMA) =====================
        if (umma::elect_one()) {
            umma::mbar_arrive_expect_tx(&w_full, (uint32_t)(2 * FB * LF_MT * 128));
            for (int b = 0; b < FB; ++b) {
                umma::tma_load_2d(smem + SM::off_w + b * (LF_MT * 128), &tmWh, &w_full, b * 64, st * LF_MT);
                umma::tma_load_2d(smem + SM::off_w + SM::W_BYTES / 2 + b * (LF_MT * 128), &tmWl, &w_full, b * 64, st * LF_MT);
            }
            int stage = 0; uint32_t phase = 0;
            for (int i = 0; i < my_blocks; ++i) {
                const int r0 = (g + i * p.groups) * LF_ROWS;
                umma::mbar_wait_guarded(&x_empty[stage], phase ^ 1);
                const bool ycopy = p.y_bulk && (int64_t)r0 + LF_ROWS <= p.N;      // full block: its 64 targets ride along
                umma::mbar_arrive_expect_tx(&x_full[stage], (uint32_t)(2 * FB * LF_ROWS * 128 + (ycopy ? SM::Y_BYTES : 0)));
                if (ycopy) bulk_copy_g2s(smem + SM::off_y + stage * SM::Y_BYTES, p.y + r0, SM::Y_BYTES, &x_full[stage]);
                uint8_t* xh = smem + SM::off_x16 + stage * SM::X16_BYTES;
                for (int b = 0; b < FB; ++b) {
                    umma::tma_load_2d(xh + b * (LF_ROWS * 128), &tmXh, &x_full[stage], b * 64, r0);
                    umma::tma_load_2d(xh + SM::X16_BYTES / 2 + b * (LF_ROWS * 128), &tmXl, &x_full[stage], b * 64, r0);
                }
                if (++stage == LF_XSTAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // ===================== logits MMA issuer: L(i) = W . X_i^T -> D1[i % 3] =====================
        // Two issuing threads (this one and warp 2), because the MMAs are small (32 / 64 tensor cycles each, 36 per block):
        // a single thread that also waits on five barriers per block was itself the critical path (~420 instructions per
        // block, 80 % busy).  All descriptors share their high word; the low word is a per-stage base plus a constant.
        if (umma::elect_one()) {
            constexpr uint32_t HI = 0x40004040u;      // SBO = 1024 B, version 1, SWIZZLE_128B
            const uint32_t idesc1 = idesc_f16_major(LF_MT, LF_ROWS, false);
            const uint32_t w_h = (umma::smem_u32(smem + SM::off_w) >> 4) | (1u << 16), w_l = w_h + (SM::W_BYTES / 2 >> 4);
            const uint32_t x0 = (umma::smem_u32(smem + SM::off_x16) >> 4) | (1u << 16);      // K-major view of X stage 0
            const int ksteps1 = KS1 > 0 ? KS1 : F / 16;
            umma::mbar_wait_guarded(&w_full, 0);
            umma::tc_fence_after();
            int xs = 0, b1 = 0;                        // X stage / D1 buffer (counters instead of i % 4, i % 3)
            uint32_t xph = 0, d1ph = 1;                // parity of x_full[xs] / d1_empty[b1] to wait for
            for (int i = 0; i < my_blocks; ++i) {
                umma::mbar_wait_guarded(&x_full[xs], xph);
                umma::mbar_wait_guarded(&d1_empty[b1], d1ph);
                umma::tc_fence_after();
                const uint32_t xk = x0 + xs * (SM::X16_BYTES >> 4);
                const uint32_t d_t = t_d1 + b1 * 64;
#pragma unroll
                for (int ks = 0; ks < (KS1 > 0 ? KS1 : 8); ++ks) {
                    if (KS1 == 0 && ks >= ksteps1) break;
                    const uint32_t ao = (ks >> 2) * (LF_MT * 128 >> 4) + (ks & 3) * 2, bo = (ks >> 2) * (LF_ROWS * 128 >> 4) + (ks & 3) * 2;
                    mma_f16_lohi(d_t, w_l + ao, xk + bo, HI, idesc1, ks != 0);
                    mma_f16_lohi(d_t, w_h + ao, xk + (SM::X16_BYTES / 2 >> 4) + bo, HI, idesc1, true);
                    mma_f16_lohi(d_t, w_h + ao, xk + bo, HI, idesc1, true);
                }
                umma::mma_commit(&d1_full[b1]);
                if (++xs == LF_XSTAGES) { xs = 0; xph ^= 1; }
                if (++b1 == LF_D1BUF) { b1 = 0; d1ph ^= 1; }
            }
        }
    } else if (warp == 2) {
        // ===================== gradient MMA issuer: D2 += d_i . X_i (X block read MN-major) =====================
        if (umma::elect_one()) {
            constexpr uint32_t HI = 0x40004040u;
            const uint32_t idesc2 = idesc_f16_major(LF_MT, F, true);
            const uint32_t d_h = (umma::smem_u32(smem + SM::off_d) >> 4) | (1u << 16), d_l = d_h + (SM::D_BYTES / 2 >> 4);
            const uint32_t x0 = (umma::smem_u32(smem + SM::off_x16) >> 4) | ((LF_ROWS * 128 >> 4) << 16);   // MN-major view: LBO = one box
            int xs = 0;
            uint32_t chain = 0;                        // index of the current D2 accumulation chain
            for (int i = 0; i < my_blocks; ++i) {
                const uint32_t buf = chain & 1;
                const bool first = (i & (LF_D2_CHAIN - 1)) == 0;
                if (first) umma::mbar_wait_guarded(&acc2_empty[buf], ((chain >> 1) & 1) ^ 1);
                umma::mbar_wait_guarded(&d_full[i & 1], (uint32_t)((i >> 1) & 1));
                umma::tc_fence_after();
                const uint32_t xm = x0 + xs * (SM::X16_BYTES >> 4);
                const uint32_t d_t = t_d2 + buf * 128;
#pragma unroll
                for (int ks = 0; ks < LF_ROWS / 16; ++ks) {
                    // A = d tile, K-major (32 bytes per k-step); B: 16 K-indices (rows of X) = 2 KB per k-step
                    if (DTMEM) {      // 16 K elements = 8 columns per k-step
                        mma_f16_ts_lohi(d_t, t_dt + 32 + ks * 8, xm + ks * 128, HI, idesc2, !first || ks != 0);
                        mma_f16_ts_lohi(d_t, t_dt + ks * 8, xm + (SM::X16_BYTES / 2 >> 4) + ks * 128, HI, idesc2, true);
                        mma_f16_ts_lohi(d_t, t_dt + ks * 8, xm + ks * 128, HI, idesc2, true);
                    } else {
                        mma_f16_lohi(d_t, d_l + ks * 2, xm + ks * 128, HI, idesc2, !first || ks != 0);
                        mma_f16_lohi(d_t, d_h + ks * 2, xm + (SM::X16_BYTES / 2 >> 4) + ks * 128, HI, idesc2, true);
                        mma_f16_lohi(d_t, d_h + ks * 2, xm + ks * 128, HI, idesc2, true);
                    }
                }
                umma::mma_commit(&x_empty[xs]);        // X block and d tile are free once these MMAs retire (the logits MMA of
                umma::mma_commit(&d_empty[i & 1]);     // this block retired long ago: d was computed from its result)
                if (!((i + 1) & (LF_D2_CHAIN - 1)) || i + 1 == my_blocks) {
                    umma::mma_commit(&acc2_full[buf]);
                    ++chain;
                }
                if (++xs == LF_XSTAGES) xs = 0;
            }
        }
    }
    } else {
        // ===================== epilogue: likelihood, d tile, D2 drains =====================
        // 16 warps = 4 per TMEM lane quarter q (vectors 32 q .. 32 q + 31 = this warp's lanes).  Two groups of 8 warps take
        // the blocks alternately (group = block parity), so one group's MUFU-heavy phase overlaps the other's ALU phase;
        // inside a group, warp half hp owns rows 32 hp .. + 31 of the block.  ALL 16 warps drain every gradient chain
        // (features 32 part .. + 31).
        asm volatile("setmaxnreg.inc.sync.aligned.u32 112;");
        const int ew = warp - LF_EPI_WARP0;
        const int q = warp & 3, part = ew >> 2, grp = part & 1, hp = part >> 1;
        const int s_local = q * 32 + lane;                          // vector inside the tile = TMEM lane = row of the d tile
        const int s_glob = st * LF_MT + s_local;
        const bool s_ok = s_glob < p.S;
        const float inv1 = 1.f / (p2_scale(*p.scal_w) * p2_scale(*p.scal_x));      // logit = D1 * inv1
        const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
        uint8_t* dh = smem + SM::off_d;
        uint8_t* dl = dh + SM::D_BYTES / 2;
        float r2[LF_EFEAT];
#pragma unroll
        for (int c = 0; c < LF_EFEAT; ++c) r2[c] = 0.f;
        double ll_total = 0.0;      // per-block fp32 sums (32 terms) are added in double: a long fp32 running sum drops the many
                                    // near-zero terms of well-classified rows once it is large (error grew linearly with N)
        uint32_t chain = 0;         // next gradient chain to drain
        auto drain = [&]() {
            const uint32_t buf = chain & 1;
            umma::mbar_wait_guarded(&acc2_full[buf], (chain >> 1) & 1);
            umma::tc_fence_after();
            float v[LF_EFEAT];
            umma::tmem_ld_32x32(t_d2 + lane_addr + buf * 128 + part * LF_EFEAT, v);
            umma::tmem_ld_wait();
#pragma unroll
            for (int c = 0; c < LF_EFEAT; ++c) r2[c] += v[c];      // round-to-nearest adds in registers
            umma::tc_fence_before();
            __syncwarp();
            if (lane == 0) umma::mbar_arrive(&acc2_empty[buf]);
            ++chain;
        };
        const int n_chains = (my_blocks + LF_D2_CHAIN - 1) / LF_D2_CHAIN;
        // Gaussian: d = r * r_scale with r_scale = p2_scale(max|y| + F max|W| max|X|) >= 2^13 / max|r|: |d| < 2^14 fits fp16
        float r_scale = 0.f;
        if constexpr (LIK == 1) r_scale = p2_scale(*p.scal_y + (float)F * *p.scal_w * *p.scal_x);
        // Cauchy: lane s owns vector s, so 1 / sigma_s is one register, loaded once
        float inv_sig = 1.f;
        if constexpr (LIK == 2) inv_sig = s_ok ? 1.f / p.sigma[s_glob] : 1.f;
        double ll2_total = 0.0;     // Cauchy: sum of z^2 / (1 + z^2)
        const uint64_t c2 = f2_pack(inv1 * 1.4426950408889634f, inv1 * 1.4426950408889634f);
        const uint64_t one2 = f2_pack(1.f, 1.f), ms2 = f2_pack(-LF_D_SCALE, -LF_D_SCALE), mone2 = f2_pack(-1.f, -1.f);
        int xs = grp % LF_XSTAGES;                     // X stage (and y slot) of this group's next block
        int b = grp;                                   // D1 buffer of this group's next block: (b + 2) % 3 per step
        uint32_t d1ph = 0;                             // parity of d1_full[b] to wait for; flips when b wraps
        const int row_step = 2 * p.groups * LF_ROWS;
        int64_t r0 = (int64_t)(g + grp * p.groups) * LF_ROWS;      // first row of this group's current block
        for (int i = grp; i < my_blocks; i += 2, r0 += row_step) {
            const int rows = (int)min((int64_t)LF_ROWS, p.N - r0);
            // targets of the block: from shared memory when they came with the X block (full block, aligned y), else lane j
            // loads y of row 32 hp + j (0 past the end of the data) before the accumulator wait and shuffles broadcast it
            const bool y_smem = p.y_bulk && rows == LF_ROWS;
            const float* ysm = reinterpret_cast<const float*>(smem + SM::off_y + xs * SM::Y_BYTES) + hp * LF_EROWS;
            xs += 2;
            if (xs >= LF_XSTAGES) xs -= LF_XSTAGES;
            float y_raw = 0.f;
            if (!y_smem) {
                const int64_t rn = r0 + hp * LF_EROWS + lane;
                y_raw = rn < p.N ? __ldg(p.y + rn) : 0.f;
            }
            umma::mbar_wait_guarded(&d1_full[b], d1ph);
            umma::tc_fence_after();
            float L[LF_EROWS];
            umma::tmem_ld_32x32(t_d1 + lane_addr + b * 64 + hp * LF_EROWS, L);
            umma::tmem_ld_wait();
            umma::tc_fence_before();
            __syncwarp();
            if (lane == 0) umma::mbar_arrive(&d1_empty[b]);
            b += 2;
            if (b >= LF_D1BUF) { b -= LF_D1BUF; d1ph ^= 1; }
            uint32_t dh_w[LF_EROWS / 2], dl_w[LF_EROWS / 2];
            float ll;                                  // Bernoulli: sum of the block's log-likelihoods; Gaussian: sum of r^2
                                                       // Cauchy: sum of log1p(z^2); Laplace: sum of |r|
            if constexpr (LIK == 0) {
                const float ys_lane = y_raw * LF_D_SCALE;
                // Per element, with raw accumulator L (logit l = L * inv1), e = exp(-|l|), sig = sigmoid(l):
                //   d * S = y S - S sig;   ll = y l - max(l, 0) - ln(1 + e)
                // summed per block as inv1 * (sum(yS L) / S - sum(max(L, 0))) - ln 2 * log2(prod(1 + e))  -- ONE log per 16 elements
                // (the product of 16 factors in (1, 2] cannot overflow), so 2 MUFU per element instead of 3.  Pairs of elements go
                // through packed fp32x2 instructions.  Rows past the end of a ragged last block have X = 0 (L = 0), where
                // d = y - 1/2 would be wrong: that block takes the predicated path.
                uint64_t acc_yl = f2_pack(0.f, 0.f), prod = one2;
                float acc_mx = 0.f;
                const uint64_t s2 = f2_pack(LF_D_SCALE, LF_D_SCALE);
                auto body = [&](auto ragged, auto from_smem) {
#pragma unroll
                    for (int k = 0; k < LF_EROWS / 2; ++k) {
                        uint64_t ys2;
                        if (decltype(from_smem)::value) {
                            const float2 yv = *reinterpret_cast<const float2*>(ysm + 2 * k);      // same address in every lane: broadcast
                            ys2 = f2_mul(f2_pack(yv.x, yv.y), s2);
                        } else {
                            ys2 = f2_pack(__shfl_sync(0xffffffffu, ys_lane, 2 * k), __shfl_sync(0xffffffffu, ys_lane, 2 * k + 1));
                        }
                        const uint64_t L2 = f2_pack(L[2 * k], L[2 * k + 1]);
                        float a0, a1, e0, e1, i0, i1, r0f, r1f;
                        f2_unpack(f2_mul(L2, c2), a0, a1);
                        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(-fabsf(a0)));
                        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(-fabsf(a1)));
                        if (decltype(ragged)::value) {
                            if (hp * LF_EROWS + 2 * k >= rows) e0 = 0.f;
                            if (hp * LF_EROWS + 2 * k + 1 >= rows) e1 = 0.f;
                        }
                        const uint64_t e2 = f2_pack(e0, e1);
                        const uint64_t ope2 = f2_add(e2, one2);
                        float o0, o1;
                        f2_unpack(ope2, o0, o1);
                        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(i0) : "f"(o0));
                        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(i1) : "f"(o1));
                        f2_unpack(f2_mul(e2, f2_pack(i0, i1)), r0f, r1f);           // sigmoid(-|l|)
                        const bool p0 = L[2 * k] >= 0.f, p1 = L[2 * k + 1] >= 0.f;
                        const uint64_t sig2 = f2_pack(p0 ? i0 : r0f, p1 ? i1 : r1f);
                        uint64_t ds2 = f2_fma(sig2, ms2, ys2);                      // S (y - sig)
                        if (p0) acc_mx += L[2 * k];
                        if (p1) acc_mx += L[2 * k + 1];
                        acc_yl = f2_fma(ys2, L2, acc_yl);
                        prod = f2_mul(prod, ope2);
                        float d0, d1;
                        f2_unpack(ds2, d0, d1);
                        if (decltype(ragged)::value) {
                            if (hp * LF_EROWS + 2 * k >= rows) d0 = 0.f;
                            if (hp * LF_EROWS + 2 * k + 1 >= rows) d1 = 0.f;
                            ds2 = f2_pack(d0, d1);
                        }
                        const __half2 h2 = __floats2half2_rn(d0, d1);
                        const float2 hfv = __half22float2(h2);
                        float l0, l1;
                        f2_unpack(f2_fma(f2_pack(hfv.x, hfv.y), mone2, ds2), l0, l1);
                        const __half2 l2 = __floats2half2_rn(l0, l1);
                        dh_w[k] = *reinterpret_cast<const uint32_t*>(&h2);
                        dl_w[k] = *reinterpret_cast<const uint32_t*>(&l2);
                    }
                };
                if (y_smem) body(std::false_type{}, std::true_type{});
                else if (rows == LF_ROWS) body(std::false_type{}, std::false_type{});
                else body(std::true_type{}, std::false_type{});
                float ay0, ay1, pr0, pr1, lg0, lg1;
                f2_unpack(acc_yl, ay0, ay1);
                f2_unpack(prod, pr0, pr1);
                asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg0) : "f"(pr0));
                asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg1) : "f"(pr1));
                ll = inv1 * ((ay0 + ay1) * (1.f / LF_D_SCALE) - acc_mx) - 0.6931471805599453f * (lg0 + lg1);
            } else if constexpr (LIK == 2) {
                // Cauchy, per element: r = y - L inv1, z = r / sigma_s, q = 1 + z^2 and ONE rcp: d = z / q lies in [-1/2, 1/2] and
                // goes out at 2^14 (the fp16 pair cannot overflow), z^2 / q adds to T.  log1p(z^2) = ln 2 (e + log2 m) with
                // q = 2^e m, m in [1, 2): the biased exponents add as integers and ONE lg2 per 16 elements takes the product of
                // 16 mantissas (< 2^16) -- the product of the factors themselves, as the Bernoulli epilogue forms it, overflows
                // here (q is unbounded).  Rows past the end of a ragged last block get r = 0: d = 0, q = 1, z^2 / q = 0.
                // (scalar instructions where a constant is involved: they take it as an immediate, a packed one needs a register
                // pair, and this epilogue is short of registers)
                const uint64_t mi2 = f2_pack(-inv1, -inv1);
                uint64_t prod = one2;
                float acc_t = 0.f;
                uint32_t esum = 0;
                auto body = [&](auto ragged, auto from_smem) {
#pragma unroll
                    for (int k = 0; k < LF_EROWS / 2; ++k) {
                        uint64_t y2;
                        if (decltype(from_smem)::value) {
                            const float2 yv = *reinterpret_cast<const float2*>(ysm + 2 * k);
                            y2 = f2_pack(yv.x, yv.y);
                        } else {
                            y2 = f2_pack(__shfl_sync(0xffffffffu, y_raw, 2 * k), __shfl_sync(0xffffffffu, y_raw, 2 * k + 1));
                        }
                        uint64_t rr2 = f2_fma(f2_pack(L[2 * k], L[2 * k + 1]), mi2, y2);
                        if (decltype(ragged)::value) {
                            float q0, q1;
                            f2_unpack(rr2, q0, q1);
                            if (hp * LF_EROWS + 2 * k >= rows) q0 = 0.f;
                            if (hp * LF_EROWS + 2 * k + 1 >= rows) q1 = 0.f;
                            rr2 = f2_pack(q0, q1);
                        }
                        float r0f, r1f, i0, i1;
                        f2_unpack(rr2, r0f, r1f);
                        const float z0 = r0f * inv_sig, z1 = r1f * inv_sig;
                        const float zz0 = z0 * z0, zz1 = z1 * z1;
                        const float o0 = zz0 + 1.f, o1 = zz1 + 1.f;
                        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(i0) : "f"(o0));
                        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(i1) : "f"(o1));
                        acc_t = __fmaf_rn(zz0, i0, acc_t);
                        acc_t = __fmaf_rn(zz1, i1, acc_t);
                        const uint32_t b0 = __float_as_uint(o0), b1 = __float_as_uint(o1);
                        esum += (b0 >> 23) + (b1 >> 23);
                        prod = f2_mul(prod, f2_pack(__uint_as_float((b0 & 0x007fffffu) | 0x3f800000u),
                                                    __uint_as_float((b1 & 0x007fffffu) | 0x3f800000u)));
                        const float d0 = z0 * i0 * (2.f * LF_D_SCALE), d1 = z1 * i1 * (2.f * LF_D_SCALE);
                        const __half2 h2 = __floats2half2_rn(d0, d1);
                        const float2 hfv = __half22float2(h2);
                        const __half2 l2 = __floats2half2_rn(d0 - hfv.x, d1 - hfv.y);
                        dh_w[k] = *reinterpret_cast<const uint32_t*>(&h2);
                        dl_w[k] = *reinterpret_cast<const uint32_t*>(&l2);
                    }
                };
                if (y_smem) body(std::false_type{}, std::true_type{});
                else if (rows == LF_ROWS) body(std::false_type{}, std::false_type{});
                else body(std::true_type{}, std::false_type{});
                float pr0, pr1, lg0, lg1;
                f2_unpack(prod, pr0, pr1);
                asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg0) : "f"(pr0));
                asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg1) : "f"(pr1));
                // every one of the 32 factors carries the exponent bias 127, padding rows (q = 1) included
                ll = 0.6931471805599453f * ((float)((int)esum - 127 * LF_EROWS) + (lg0 + lg1));
                ll2_total += (double)acc_t;
            } else if constexpr (LIK == 3) {
                // Laplace, per element: r = y - L inv1, d = sign(r) (sign(0) = 0, as torch's abs gradient), exact in fp16 at 2^13
                // with a zero lo word; |r| adds to A.  No MUFU op.  Rows past the end of a ragged last block get r = 0: d = 0.
                const uint64_t mi2 = f2_pack(-inv1, -inv1);
                float acc_a0 = 0.f, acc_a1 = 0.f;
                auto body = [&](auto ragged, auto from_smem) {
#pragma unroll
                    for (int k = 0; k < LF_EROWS / 2; ++k) {
                        uint64_t y2;
                        if (decltype(from_smem)::value) {
                            const float2 yv = *reinterpret_cast<const float2*>(ysm + 2 * k);
                            y2 = f2_pack(yv.x, yv.y);
                        } else {
                            y2 = f2_pack(__shfl_sync(0xffffffffu, y_raw, 2 * k), __shfl_sync(0xffffffffu, y_raw, 2 * k + 1));
                        }
                        float q0, q1;
                        f2_unpack(f2_fma(f2_pack(L[2 * k], L[2 * k + 1]), mi2, y2), q0, q1);
                        if (decltype(ragged)::value) {
                            if (hp * LF_EROWS + 2 * k >= rows) q0 = 0.f;
                            if (hp * LF_EROWS + 2 * k + 1 >= rows) q1 = 0.f;
                        }
                        acc_a0 += fabsf(q0);
                        acc_a1 += fabsf(q1);
                        const float d0 = q0 > 0.f ? LF_D_SCALE : (q0 < 0.f ? -LF_D_SCALE : 0.f);
                        const float d1 = q1 > 0.f ? LF_D_SCALE : (q1 < 0.f ? -LF_D_SCALE : 0.f);
                        const __half2 h2 = __floats2half2_rn(d0, d1);
                        dh_w[k] = *reinterpret_cast<const uint32_t*>(&h2);
                        dl_w[k] = 0u;
                    }
                };
                if (y_smem) body(std::false_type{}, std::true_type{});
                else if (rows == LF_ROWS) body(std::false_type{}, std::false_type{});
                else body(std::true_type{}, std::false_type{});
                ll = acc_a0 + acc_a1;
            } else {
                // r = y - L inv1 per element (no MUFU op); rows past the end of a ragged last block get r = 0
                const uint64_t mi2 = f2_pack(-inv1, -inv1), rs2 = f2_pack(r_scale, r_scale);
                uint64_t acc_rr = f2_pack(0.f, 0.f);
                auto body = [&](auto ragged, auto from_smem) {
#pragma unroll
                    for (int k = 0; k < LF_EROWS / 2; ++k) {
                        uint64_t y2;
                        if (decltype(from_smem)::value) {
                            const float2 yv = *reinterpret_cast<const float2*>(ysm + 2 * k);
                            y2 = f2_pack(yv.x, yv.y);
                        } else {
                            y2 = f2_pack(__shfl_sync(0xffffffffu, y_raw, 2 * k), __shfl_sync(0xffffffffu, y_raw, 2 * k + 1));
                        }
                        uint64_t rr2 = f2_fma(f2_pack(L[2 * k], L[2 * k + 1]), mi2, y2);
                        if (decltype(ragged)::value) {
                            float q0, q1;
                            f2_unpack(rr2, q0, q1);
                            if (hp * LF_EROWS + 2 * k >= rows) q0 = 0.f;
                            if (hp * LF_EROWS + 2 * k + 1 >= rows) q1 = 0.f;
                            rr2 = f2_pack(q0, q1);
                        }
                        acc_rr = f2_fma(rr2, rr2, acc_rr);
                        const uint64_t ds2 = f2_mul(rr2, rs2);
                        float d0, d1;
                        f2_unpack(ds2, d0, d1);
                        const __half2 h2 = __floats2half2_rn(d0, d1);
                        const float2 hfv = __half22float2(h2);
                        float l0, l1;
                        f2_unpack(f2_fma(f2_pack(hfv.x, hfv.y), f2_pack(-1.f, -1.f), ds2), l0, l1);
                        const __half2 l2 = __floats2half2_rn(l0, l1);
                        dh_w[k] = *reinterpret_cast<const uint32_t*>(&h2);
                        dl_w[k] = *reinterpret_cast<const uint32_t*>(&l2);
                    }
                };
                if (y_smem) body(std::false_type{}, std::true_type{});
                else if (rows == LF_ROWS) body(std::false_type{}, std::false_type{});
                else body(std::true_type{}, std::false_type{});
                float a0, a1;
                f2_unpack(acc_rr, a0, a1);
                ll = a0 + a1;
            }
            // the d tile is free once the gradient MMA of the previous block (the other group's) has retired
            // (block i - 1: barrier of the other parity, its use (i - 1) / 2; the first block has nothing to wait for)
            if (i > 0) umma::mbar_wait_guarded(&d_empty[(i & 1) ^ 1], (uint32_t)(((i - 1) >> 1) & 1));
            if (DTMEM) {
                // this thread owns TMEM lane s_local = row s of the A operand; column = pair of block rows (2k, 2k + 1)
                umma::tc_fence_after();
                tmem_st_32x16(t_dt + lane_addr + hp * (LF_EROWS / 2), dh_w);
                tmem_st_32x16(t_dt + 32 + lane_addr + hp * (LF_EROWS / 2), dl_w);
                tmem_st_wait();
                umma::tc_fence_before();
            } else {
            // K-major A tile [128 vectors][64 rows] fp16, 128-byte rows, SWIZZLE_128B: this thread owns row s_local and writes
            // the 4 chunks (8 rows of X each) of its rows
#pragma unroll
            for (int cc = 0; cc < LF_EROWS / 8; ++cc) {
                const int c = hp * (LF_EROWS / 8) + cc;
                const int off = s_local * 128 + ((c ^ (s_local & 7)) << 4);
                *reinterpret_cast<uint4*>(dh + off) = make_uint4(dh_w[4 * cc], dh_w[4 * cc + 1], dh_w[4 * cc + 2], dh_w[4 * cc + 3]);
                *reinterpret_cast<uint4*>(dl + off) = make_uint4(dl_w[4 * cc], dl_w[4 * cc + 1], dl_w[4 * cc + 2], dl_w[4 * cc + 3]);
            }
            umma::fence_proxy_async();
            }
            ll_total += (double)ll;
            __syncwarp();
            if (lane == 0) umma::mbar_arrive(&d_full[grp]);
            // chains that ended at or before block i - 1 are complete (or about to be): drain them now, while the tensor core
            // works on this block's d  (chain c covers blocks 2c, 2c + 1)
            while ((int)chain < n_chains && (int)(chain * LF_D2_CHAIN + LF_D2_CHAIN - 1) < i) drain();
        }
        while ((int)chain < n_chains) drain();
        // this CTA's share of + d ll / d W for vector s_glob, features 32 part .. + 31
        if (s_ok) {
            constexpr float d_scale = LIK == 2 ? 2.f * LF_D_SCALE : LF_D_SCALE;      // Cauchy: |d| <= 1/2 goes out at 2^14
            const float inv2 = 1.f / ((LIK == 1 ? r_scale : d_scale) * p2_scale(*p.scal_x));
            float* o = p.part + (int64_t)g * p.part_stride + (int64_t)s_glob * F + part * LF_EFEAT;
#pragma unroll
            for (int c = 0; c < LF_EFEAT; c += 4)
                if (part * LF_EFEAT + c < F)
                    *reinterpret_cast<float4*>(o + c) = make_float4(r2[c] * inv2, r2[c + 1] * inv2, r2[c + 2] * inv2, r2[c + 3] * inv2);
        }
        if constexpr (LIK != 0) {
            // lane s owns vector s: the two epilogue groups and two row halves of this CTA and every row group add to R[s]
            if (s_ok && ll_total != 0.0) atomicAdd(p.R + s_glob, ll_total);
            if constexpr (LIK == 2)
                if (s_ok && ll2_total != 0.0) atomicAdd(p.T + s_glob, ll2_total);
        } else {
        double tot = s_ok ? ll_total : 0.0;      // vectors past S are zero rows of the W tile: their terms are not part of the sum
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, o);
        if (lane == 0 && tot != 0.0) atomicAdd(p.loss, tot * (double)p.loss_scale);
        }
    }
    umma::tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        umma::tc_fence_after();
        umma::tmem_dealloc(tmem_base, 512);
    }
}

// x [n] fp32 -> fp16 (hi, lo) pair of x * p2_scale(*bound)   (n % 8 == 0, x and the outputs 16-byte aligned)
__global__ void __launch_bounds__(256)
linear_flash_split_kernel(const float* __restrict__ x, int64_t n, const float* __restrict__ bound, __half* __restrict__ hi,
                          __half* __restrict__ lo) {
    const float sc = p2_scale(*bound);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n / 8; q += stride) {
        const float4 a = __ldcs(reinterpret_cast<const float4*>(x) + 2 * q);
        const float4 b = __ldcs(reinterpret_cast<const float4*>(x) + 2 * q + 1);
        const float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        uint32_t hh[4], ll[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float x0 = v[2 * k] * sc, x1 = v[2 * k + 1] * sc;
            const __half2 h2 = __floats2half2_rn(x0, x1);
            const float2 hf = __half22float2(h2);
            const __half2 l2 = __floats2half2_rn(x0 - hf.x, x1 - hf.y);
            hh[k] = *reinterpret_cast<const uint32_t*>(&h2);
            ll[k] = *reinterpret_cast<const uint32_t*>(&l2);
        }
        reinterpret_cast<uint4*>(hi)[q] = make_uint4(hh[0], hh[1], hh[2], hh[3]);
        reinterpret_cast<uint4*>(lo)[q] = make_uint4(ll[0], ll[1], ll[2], ll[3]);
    }
}

// slot = max(slot, max |x|) (non-negative floats order like their bit patterns); one atomic per block
__global__ void __launch_bounds__(256) lf_absmax_kernel(const float* __restrict__ x, int64_t n, float* __restrict__ slot) {
    __shared__ float red[8];
    float m = 0.f;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if ((reinterpret_cast<uintptr_t>(x) & 15) == 0) {
        const float4* x4 = reinterpret_cast<const float4*>(x);
        for (int64_t q = i0; q < n / 4; q += stride) {
            const float4 v = __ldg(x4 + q);
            m = fmaxf(fmaxf(m, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
        }
        for (int64_t j = n / 4 * 4 + i0; j < n; j += stride) m = fmaxf(m, fabsf(x[j]));
    } else {
        for (int64_t i = i0; i < n; i += stride) m = fmaxf(m, fabsf(x[i]));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = red[0];
        for (int w = 1; w < 8; ++w) t = fmaxf(t, red[w]);
        if (t > 0.f) atomicMax(reinterpret_cast<unsigned int*>(slot), __float_as_uint(t));
    }
}

struct LinearFlashBuffers {
    __half *Wh, *Wl;       // [S][F] fp16 pair
    __half *Xh, *Xl;       // [N][F] fp16 pair (set by the owner: aliases the staged variant's fp32 pair buffers)
    float* scal;           // 64 floats, zeroed per call
    float* part;           // [groups][S][F]
    int groups, tiles;
    template <class Take>
    void carve(Take&& take, int S, int F, int sms) {
        tiles = (S + LF_MT - 1) / LF_MT;
        groups = sms / tiles;
        if (groups < 1) groups = 1;
        Wh = reinterpret_cast<__half*>(take(((size_t)S * F + 1) / 2));
        Wl = reinterpret_cast<__half*>(take(((size_t)S * F + 1) / 2));
        scal = take(64);
        part = take((size_t)groups * S * F);
    }
};

static bool linear_flash_ok(const float* X, int64_t N, int F, int S) {
    if (const char* env = getenv("BRN_LINEAR_FLASH"))
        if (!atoi(env)) return false;
    return N >= 1 && N < (int64_t)1 << 31 && S >= 1 && F % 16 == 0 && F <= LF_FMAX && (reinterpret_cast<uintptr_t>(X) & 15) == 0;
}

// A prepared X: [64 floats: [0] = max |X|] [Xh: N * F fp16] [Xl: N * F fp16]  (brn_linear_prepare_x)
constexpr size_t LF_PX_HEADER = 256;
static size_t linear_prepared_x_bytes(int64_t N, int F) {
    if (N < 1 || N >= (int64_t)1 << 31 || F % 16 != 0 || F > LF_FMAX || F < 16) return 0;
    return LF_PX_HEADER + 2 * ((size_t)N * F * 2 + 255) / 256 * 256;
}
static __half* prepared_x_hi(const void* px) { return reinterpret_cast<__half*>(const_cast<char*>(static_cast<const char*>(px)) + LF_PX_HEADER); }
static __half* prepared_x_lo(const void* px, int64_t N, int F) {
    return reinterpret_cast<__half*>(const_cast<char*>(static_cast<const char*>(px)) + LF_PX_HEADER + ((size_t)N * F * 2 + 255) / 256 * 256);
}
// max |X| and the scaled fp16 (hi, lo) pair of X: one read for the bound, one read + one write of X's own size for the pair
static int launch_prepare_x(const float* X, int64_t N, int F, float* bound, __half* hi, __half* lo, cudaStream_t stream) {
    BRN_CUDA_OK(cudaMemsetAsync(bound, 0, sizeof(float), stream));
    lf_absmax_kernel<<<(unsigned)std::min<int64_t>((N * F / 4 + 255) / 256 + 1, 1184), 256, 0, stream>>>(X, N * F, bound);
    BRN_LAUNCH_OK("lf_absmax_kernel");
    linear_flash_split_kernel<<<(unsigned)std::min<int64_t>((N * F / 8 + 255) / 256 + 1, 2368), 256, 0, stream>>>(X, N * F, bound, hi, lo);
    BRN_LAUNCH_OK("linear_flash_split_kernel");
    return 0;
}

// dW [S][F] = + d ll / d W, loss += loss_scale * sum ll for S weight vectors W [S][F] over N rows (Bernoulli, C == 1).
// px: a prepared X (the caller keeps it while X does not change: a training loop over fixed data then reads X once per
// evaluation, as fp16 pairs, instead of three times), or NULL: X is split into the workspace on every call.
// R != NULL selects a regression epilogue, lik (the LIK codes of linear_flash_kernel): 1 = Gaussian, the per-slice partials of
// G_s = sum_b r_sb x_b, r_sb = y_b - w_s . x_b, go to b.part and R[s] += sum_b r_sb^2 (loss is unused); 2 = Cauchy, with the
// noise scales sigma [S]: G_s = sum_b z/(1 + z^2) x_b, z = r_sb / sigma_s, R[s] += sum_b log1p(z^2), T[s] += sum_b z^2/(1 + z^2);
// 3 = Laplace: G_s = sum_b sign(r_sb) x_b, R[s] += sum_b |r_sb|.
static int launch_linear_flash(const float* X, const void* px, const float* y, int64_t N, int F, int S, const float* W, float* dW,
                               float loss_scale, double* loss, const LinearFlashBuffers& b, cudaStream_t stream,
                               double* R = nullptr, int lik = 1, const float* sigma = nullptr, double* T = nullptr) {
    BRN_CUDA_OK(cudaMemsetAsync(b.scal, 0, 64 * sizeof(float), stream));
    lf_absmax_kernel<<<(unsigned)std::min<int64_t>(((int64_t)S * F / 4 + 255) / 256 + 1, 148), 256, 0, stream>>>(W, (int64_t)S * F, b.scal);
    BRN_LAUNCH_OK("lf_absmax_kernel");
    linear_flash_split_kernel<<<(unsigned)std::min<int64_t>(((int64_t)S * F / 8 + 255) / 256 + 1, 1184), 256, 0, stream>>>(
        W, (int64_t)S * F, b.scal, b.Wh, b.Wl);
    BRN_LAUNCH_OK("linear_flash_split_kernel");
    const __half *Xh = b.Xh, *Xl = b.Xl;
    const float* scal_x = b.scal + 1;
    if (px) {
        Xh = prepared_x_hi(px); Xl = prepared_x_lo(px, N, F); scal_x = static_cast<const float*>(px);
    } else if (int e = launch_prepare_x(X, N, F, b.scal + 1, b.Xh, b.Xl, stream)) {
        return e;
    }
    if (R && lik == 1) {
        lf_absmax_kernel<<<(unsigned)std::min<int64_t>((N / 4 + 255) / 256 + 1, 148), 256, 0, stream>>>(y, N, b.scal + 2);
        BRN_LAUNCH_OK("lf_absmax_kernel");
    }
    CUtensorMap tWh, tWl, tXh, tXl;
    if (int e = make_tmap_2d_f16(&tWh, b.Wh, S, F, F, LF_MT, 64)) return e;
    if (int e = make_tmap_2d_f16(&tWl, b.Wl, S, F, F, LF_MT, 64)) return e;
    if (int e = make_tmap_2d_f16(&tXh, Xh, N, F, F, LF_ROWS, 64)) return e;
    if (int e = make_tmap_2d_f16(&tXl, Xl, N, F, F, LF_ROWS, 64)) return e;
    LinearFlashParams p;
    p.y = y; p.N = N; p.F = F; p.S = S; p.scal_w = b.scal; p.scal_x = scal_x; p.part = b.part; p.part_stride = (int64_t)S * F;
    p.loss = loss; p.loss_scale = loss_scale; p.groups = b.groups;
    p.scal_y = b.scal + 2; p.R = R;
    p.sigma = sigma; p.T = T;
    p.y_bulk = (reinterpret_cast<uintptr_t>(y) & 15) == 0;
    if (const char* env = getenv("BRN_LINEAR_Y_BULK")) p.y_bulk = p.y_bulk && atoi(env) != 0;
    dim3 grid(b.tiles, b.groups);
    int dtmem = 1;
    if (const char* env = getenv("BRN_LINEAR_DTMEM")) dtmem = atoi(env) != 0;
    auto launch = [&](auto kern, int smem_bytes) -> int {
        BRN_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
        kern<<<grid, LF_THREADS, smem_bytes, stream>>>(tWh, tWl, tXh, tXl, p);
        return 0;
    };
    if (R && lik == 2) {      // the regression epilogues exist with the d tile in tensor memory only
        if (int e = F == 128 ? launch(linear_flash_kernel<8, 1, 2>, LinearFlashSmem<1>::TOTAL)
                             : launch(linear_flash_kernel<0, 1, 2>, LinearFlashSmem<1>::TOTAL))
            return e;
    } else if (R && lik == 3) {
        if (int e = F == 128 ? launch(linear_flash_kernel<8, 1, 3>, LinearFlashSmem<1>::TOTAL)
                             : launch(linear_flash_kernel<0, 1, 3>, LinearFlashSmem<1>::TOTAL))
            return e;
    } else if (R) {
        if (int e = F == 128 ? launch(linear_flash_kernel<8, 1, 1>, LinearFlashSmem<1>::TOTAL)
                             : launch(linear_flash_kernel<0, 1, 1>, LinearFlashSmem<1>::TOTAL))
            return e;
    } else if (F == 128) {
        if (int e = dtmem ? launch(linear_flash_kernel<8, 1>, LinearFlashSmem<1>::TOTAL) : launch(linear_flash_kernel<8, 0>, LinearFlashSmem<0>::TOTAL)) return e;
    } else {
        if (int e = dtmem ? launch(linear_flash_kernel<0, 1>, LinearFlashSmem<1>::TOTAL) : launch(linear_flash_kernel<0, 0>, LinearFlashSmem<0>::TOTAL)) return e;
    }
    BRN_LAUNCH_OK("linear_flash_kernel");
    return 0;
}

}  // namespace brn
