// tcgen05 "NT" GEMM with 3xTF32 split for fp32-equivalent accuracy:
//     D[m, n] = sum_k A[m, k] * B[n, k]            A: [M][K], B: [N][K], both K-contiguous ("K-major")
// Operands arrive pre-split in HBM as TF32-exact pairs (hi, lo) -- see umma::split_tf32 -- and are moved
// by TMA (128-byte swizzle) into a multi-stage shared-memory ring; one elected thread issues
//     D += A_lo.B_hi^T ; D += A_hi.B_lo^T ; D += A_hi.B_hi^T      (tcgen05.mma kind::tf32, M=128, N=BN, K=8)
// accumulating in TMEM.  Persistent: each CTA walks a list of (m-tile, n-tile) units; TMA producer, MMA
// issuer and epilogue are separate warps synchronised only by mbarriers.
//
// Accuracy: the tensor core TRUNCATES (round-toward-zero) its fp32 accumulator after every instruction
// (measured on B200: relative bias -2.7e-8 .. -5e-8 per MMA, i.e. -1e-5 after K=1024), which is outside the
// 1e-5 parity budget.  The accumulation chain in TMEM is therefore kept short: every `drain_chunks` K chunks
// the MMA warp switches to the other of two TMEM accumulator buffers and the epilogue warps drain the
// finished one into fp32 REGISTERS with round-to-nearest adds, fully overlapped with the next block's MMAs.
#pragma once
#include "common.cuh"
#include "umma.cuh"
#include <type_traits>

namespace brn {

constexpr int UG_BM = 128;        // rows of A per tile (TMEM lanes)
// BK = fp32 elements per K chunk = one swizzle row: 32 (128 B, 2-stage ring) or 16 (64 B swizzle, 5-stage ring).  The
// finer chunk keeps 4 loads in flight while one is consumed: the 2-stage ring left the tensor pipe idle ~35 % of the
// time waiting for the next 86 KB stage (ncu: profiles/r1a_*), the 5-stage ring hides that latency.
constexpr int UG_BUF_COLS = 256;  // TMEM column stride between the two accumulator buffers
constexpr int UG_EPI_WARPS = 8;   // epilogue warps: 4 TMEM lane quarters x 2 column halves

// an epilogue policy may declare `static constexpr bool TRANSFORMS_A = true` together with transform_a_context(params) ->
// float and transform_a(ctx, x) -> float: the converter warps of a SPLIT & 1 kernel then map every A element before
// splitting it
template <class Epi, class = void>
struct epi_transforms_a : std::false_type {};
template <class Epi>
struct epi_transforms_a<Epi, std::void_t<decltype(Epi::TRANSFORMS_A)>> : std::bool_constant<Epi::TRANSFORMS_A> {};

template <int BN, int BK>
struct UmmaSmem {
    static constexpr int A_BYTES = UG_BM * BK * 4;
    static constexpr int B_BYTES = BN * BK * 4;
    static constexpr int STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;
    static constexpr int MAX_STAGES = (227 * 1024 - 1024) / STAGE_BYTES;
    static constexpr int STAGES = MAX_STAGES >= 5 ? 5 : MAX_STAGES;       // e.g. BN=208/BK=16: 5, BN=256/BK=16: 4, BN=128/BK=32: 3
    static_assert(STAGES >= 2, "tile too large for a double-buffered ring");
    static constexpr int TOTAL = STAGES * STAGE_BYTES + 1024;   // + alignment slack
    static_assert(A_BYTES % (8 * BK * 4) == 0 && B_BYTES % (8 * BK * 4) == 0, "tiles must be whole swizzle atoms");
};

// which (m-tile, n-tile, K range) units a CTA processes, identically enumerated by every warp role.
// mode 0: units n-major (concurrently running CTAs share the B tile), round-robin over CTAs.  When the last round
//         would be nearly empty (T = units % grid <= grid/2) those T tail units are instead SPLIT ALONG K over the whole
//         grid (J = grid/T slices each) and accumulated with atomics into a caller-zeroed output: a [7 x 128]-unit
//         problem on 148 CTAs costs 6 + 1/J unit-times instead of 7.
// mode 1: a CTA keeps its m-tile and strides over n-tiles.
// mode 2: units m-major (concurrently running CTAs share the A tile: tall-skinny problems whose A operand is the large
//         one, e.g. [rows x features] activations against a small weight matrix), round-robin, no K split.
struct UnitIter {
    int m_tiles, n_tiles, k_chunks, mode;
    int u, step, end, mt_fixed;
    int tail_u, tail_j, J;
    bool has_tail;
    __device__ UnitIter(int m_tiles_, int n_tiles_, int k_chunks_, int mode_, int split_T, int full_units)
        : m_tiles(m_tiles_), n_tiles(n_tiles_), k_chunks(k_chunks_), mode(mode_), tail_u(0), tail_j(0), J(1), has_tail(false) {
        if (mode == 0 || mode == 2) {
            u = blockIdx.x; step = gridDim.x; end = m_tiles * n_tiles; mt_fixed = -1;
            if (split_T > 0) {
                end = full_units;
                J = min((int)gridDim.x / split_T, k_chunks);
                has_tail = (int)blockIdx.x < split_T * J;
                tail_u = full_units + (int)blockIdx.x % split_T;
                tail_j = (int)blockIdx.x / split_T;
            }
        } else {
            mt_fixed = blockIdx.x % m_tiles;
            int g = blockIdx.x / m_tiles, G = gridDim.x / m_tiles;
            u = g; step = G; end = (g < G) ? n_tiles : 0;
        }
    }
    __device__ bool in_tail() const { return u >= end; }
    __device__ bool valid() const { return u < end || has_tail; }
    __device__ void next() {
        if (u < end) u += step;
        else has_tail = false;
    }
    __device__ int unit() const { return u < end ? u : tail_u; }
    __device__ int mt() const { return mode == 0 ? unit() % m_tiles : (mode == 2 ? unit() / n_tiles : mt_fixed); }
    __device__ int nt() const { return mode == 0 ? unit() / m_tiles : (mode == 2 ? unit() % n_tiles : u); }
    __device__ int slice() const { return u < end ? 0 : tail_j; }
    __device__ int kc_begin() const { return u < end ? 0 : (int)((long long)tail_j * k_chunks / J); }
    __device__ int kc_end() const { return u < end ? k_chunks : (int)((long long)(tail_j + 1) * k_chunks / J); }
};

// EW = epilogue warps (8 or 16): 4 TMEM lane quarters x EW/4 column blocks of CPT = BN / (EW/4) columns.  16 warps halve the
// per-thread register footprint (BN = 256 becomes possible) and double the issue-level parallelism of a heavy epilogue.
// SPLIT_A: the A operand arrives as ONE plain fp32 matrix (tensor map tmAh; tmAl unused).  TMA drops the fp32 tile into the
// A_hi slot of the stage and four converter warps split it in place -- hi = rn_tf32(x) stays, lo = rn_tf32(x - hi) goes to
// the same (swizzled) offset of the A_lo slot -- before the MMA warp may read the stage.  An operand that is produced by a
// previous kernel and consumed once (K2: d = y - sigmoid(l)) then crosses HBM as 4 instead of 8 bytes per element.
// SPLIT is a bit mask: 1 = the A operand, 2 = the B operand arrives plain (tensor map tmBh; tmBl unused).
// CW = converter warps (2 keep a 16-epilogue-warp kernel at 640 threads = 96 registers per thread).
// KIND: 0 = tf32 operands (fp32 words, 3xTF32), 1 = fp16 operands (hi / lo halves, "3xFP16": the same 11 + 11 mantissa bits
// per operand as the TF32 pair at twice the MACs per instruction and half the operand bytes; the caller pre-scales the
// operands by powers of two into the fp16 range and un-scales in the epilogue).  BK counts 32-bit words per chunk row.
// MAJOR: 0 = both operands K-major (A [M][K], B [N][K]); 1 = both MN-major (A [K][M], B [K][N], i.e. D = A^T B for two
// row-major matrices that share their ROW index as the contraction index -- a weight gradient sum_r d[r, m] a[r, n] read
// straight from the row-major activations, no transposed copies).  MN-major stages hold BM/32 resp. BN/32 TMA boxes of
// [BK rows][32 columns] (SWIZZLE_128B); tf32 operands only.
template <int BN, int BK, class Epi, int EW = UG_EPI_WARPS, int SPLIT = 0, int CW = 4, int KIND = 0, int MAJOR = 0>
__global__ void __launch_bounds__(64 + 32 * EW + (SPLIT ? 32 * CW : 0), 1)
umma_nt_3xtf32_kernel(const __grid_constant__ CUtensorMap tmAh, const __grid_constant__ CUtensorMap tmAl,
                      const __grid_constant__ CUtensorMap tmBh, const __grid_constant__ CUtensorMap tmBl,
                      int m_tiles, int n_tiles, int k_chunks, int drain_chunks, int mode, int split_T, int full_units,
                      typename Epi::Params ep) {
    using SM = UmmaSmem<BN, BK>;
    constexpr int UG_STAGES = SM::STAGES, UG_BK = BK, SW = BK * 4;
    constexpr bool SPLIT_A = (SPLIT & 1) != 0, SPLIT_B = (SPLIT & 2) != 0;
    constexpr int UG_CONV_WARPS = CW;
    constexpr int CPT = BN / (EW / 4);             // accumulator columns per epilogue thread
    static_assert(EW == 4 || EW == 8 || EW == 16, "4, 8 or 16 epilogue warps");
    static_assert(KIND == 0 || SPLIT == 0, "on-the-fly operand splitting exists for tf32 operands only");
    static_assert(MAJOR == 0 || (KIND == 0 && BN % 32 == 0 && BK % 8 == 0), "MN-major operands: tf32, N tile a multiple of 32 columns");
    constexpr int KE = KIND == 0 ? 1 : 2;          // operand elements per 32-bit word
    static_assert(BN <= UG_BUF_COLS && BN % 16 == 0 && CPT % 8 == 0, "unsupported N tile");
    constexpr uint32_t TMEM_COLS = 512;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    __shared__ __align__(8) uint64_t full_bar[UG_STAGES], empty_bar[UG_STAGES], acc_full[2], acc_empty[2];
    __shared__ __align__(8) uint64_t conv_bar[SPLIT ? UG_STAGES : 1];       // stage converted (SPLIT_A): UG_CONV_WARPS arrivals
    __shared__ uint32_t tmem_base_slot;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        umma::tma_prefetch_desc(&tmAh); umma::tma_prefetch_desc(&tmAl);
        umma::tma_prefetch_desc(&tmBh); umma::tma_prefetch_desc(&tmBl);
        for (int s = 0; s < UG_STAGES; ++s) { umma::mbar_init(&full_bar[s], 1); umma::mbar_init(&empty_bar[s], 1); }
        for (int b = 0; b < 2; ++b) { umma::mbar_init(&acc_full[b], 1); umma::mbar_init(&acc_empty[b], EW); }
        if (SPLIT)
            for (int s = 0; s < UG_STAGES; ++s) umma::mbar_init(&conv_bar[s], UG_CONV_WARPS);
        umma::fence_barrier_init();
    }
    if (warp == 1) umma::tmem_alloc(&tmem_base_slot, TMEM_COLS);
    umma::tc_fence_before();
    __syncthreads();
    umma::tc_fence_after();
    const uint32_t tmem_base = tmem_base_slot;

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (umma::elect_one()) {
            int stage = 0; uint32_t phase = 0;
            for (UnitIter it(m_tiles, n_tiles, k_chunks, mode, split_T, full_units); it.valid(); it.next()) {
                const int m0 = it.mt() * UG_BM, n0 = it.nt() * BN;
                const int kcb = it.kc_begin(), kce = it.kc_end();
                for (int kc = kcb; kc < kce; ++kc) {
                    umma::mbar_wait(&empty_bar[stage], phase ^ 1);
                    uint8_t* st = smem + stage * SM::STAGE_BYTES;
                    umma::mbar_arrive_expect_tx(&full_bar[stage], SM::STAGE_BYTES - (SPLIT_B ? SM::B_BYTES : 0) -
                                                                      (SPLIT_A ? SM::A_BYTES : 0));
                    const int k0 = kc * UG_BK * KE;
                    if constexpr (MAJOR == 1) {
                        // boxes of [BK rows of K][32 columns of M / N]; columns past the matrix are zero-filled
                        constexpr int BOX = UG_BK * 128;
                        for (int b = 0; b < UG_BM / 32; ++b) {
                            umma::tma_load_2d(st + b * BOX, &tmAh, &full_bar[stage], m0 + 32 * b, k0);
                            if (!SPLIT_A) umma::tma_load_2d(st + SM::A_BYTES + b * BOX, &tmAl, &full_bar[stage], m0 + 32 * b, k0);
                        }
                        for (int b = 0; b < BN / 32; ++b) {
                            umma::tma_load_2d(st + 2 * SM::A_BYTES + b * BOX, &tmBh, &full_bar[stage], n0 + 32 * b, k0);
                            if (!SPLIT_B)
                                umma::tma_load_2d(st + 2 * SM::A_BYTES + SM::B_BYTES + b * BOX, &tmBl, &full_bar[stage], n0 + 32 * b, k0);
                        }
                    } else {
                    umma::tma_load_2d(st, &tmAh, &full_bar[stage], k0, m0);
                    if (!SPLIT_A) umma::tma_load_2d(st + SM::A_BYTES, &tmAl, &full_bar[stage], k0, m0);
                    umma::tma_load_2d(st + 2 * SM::A_BYTES, &tmBh, &full_bar[stage], k0, n0);
                    if (!SPLIT_B)
                        umma::tma_load_2d(st + 2 * SM::A_BYTES + SM::B_BYTES, &tmBl, &full_bar[stage], k0, n0);
                    }
                    if (++stage == UG_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        if (umma::elect_one()) {      // not `lane == 0`: ptxas then issues each UTCHMMA once instead of inside an ELECT loop
            constexpr uint32_t idesc = MAJOR == 1 ? umma::idesc_tf32_mn(UG_BM, BN) : umma::idesc_kind<KIND>(UG_BM, BN);
            int stage = 0; uint32_t phase = 0, blk = 0;
            for (UnitIter it(m_tiles, n_tiles, k_chunks, mode, split_T, full_units); it.valid(); it.next()) {
                const int kcb = it.kc_begin(), kce = it.kc_end();
                for (int kc0 = kcb; kc0 < kce; kc0 += drain_chunks, ++blk) {
                    const uint32_t buf = blk & 1, use = (blk >> 1) & 1;
                    umma::mbar_wait(&acc_empty[buf], use ^ 1);     // epilogue has drained this buffer's previous use
                    umma::tc_fence_after();
                    const uint32_t d_tmem = tmem_base + buf * UG_BUF_COLS;
                    const int kc1 = min(kc0 + drain_chunks, kce);
                    for (int kc = kc0; kc < kc1; ++kc) {
                        umma::mbar_wait(SPLIT ? &conv_bar[stage] : &full_bar[stage], phase);
                        umma::tc_fence_after();
                        const uint32_t st = umma::smem_u32(smem + stage * SM::STAGE_BYTES);
                        const uint32_t ah = st, al = st + SM::A_BYTES, bh = st + 2 * SM::A_BYTES, bl = bh + SM::B_BYTES;
#pragma unroll
                        for (int ks = 0; ks < UG_BK / 8; ++ks) {
                            // MN-major: LBO = one box, SBO = one 4-row atom (512 B), 8 K indices per MMA = two atoms = 1024 B
                            constexpr uint32_t BOX = UG_BK * 128, SBO_ = 512;
                            const uint32_t ko = MAJOR == 1 ? ks * 1024 : ks * 32;   // K-major: 8 tf32 = 32 bytes along the swizzle row
                            const uint64_t dah = MAJOR == 1 ? umma::smem_desc_mn(ah + ko, BOX, SBO_, 1) : umma::smem_desc_k<SW>(ah + ko);
                            const uint64_t dal = MAJOR == 1 ? umma::smem_desc_mn(al + ko, BOX, SBO_, 1) : umma::smem_desc_k<SW>(al + ko);
                            const uint64_t dbh = MAJOR == 1 ? umma::smem_desc_mn(bh + ko, BOX, SBO_, 1) : umma::smem_desc_k<SW>(bh + ko);
                            const uint64_t dbl = MAJOR == 1 ? umma::smem_desc_mn(bl + ko, BOX, SBO_, 1) : umma::smem_desc_k<SW>(bl + ko);
                            umma::mma_ss<KIND>(d_tmem, dal, dbh, idesc, kc != kc0 || ks != 0);
                            umma::mma_ss<KIND>(d_tmem, dah, dbl, idesc, true);
                            umma::mma_ss<KIND>(d_tmem, dah, dbh, idesc, true);
                        }
                        umma::mma_commit(&empty_bar[stage]);       // smem stage reusable once these MMAs retire
                        if (++stage == UG_STAGES) { stage = 0; phase ^= 1; }
                    }
                    umma::mma_commit(&acc_full[buf]);
                }
            }
        }
    } else if (SPLIT && warp >= 2 + EW) {
        // ===================== converter warps (SPLIT_A) =====================
        // 128 threads, A_BYTES / 16 float4 per stage; element-wise and in place, so the swizzle TMA applied is irrelevant
        const int ct = threadIdx.x - 32 * (2 + EW);
        float a_ctx = 0.f;
        if constexpr (epi_transforms_a<Epi>::value) a_ctx = Epi::transform_a_context(ep);
        (void)a_ctx;
        int stage = 0; uint32_t phase = 0;
        for (UnitIter it(m_tiles, n_tiles, k_chunks, mode, split_T, full_units); it.valid(); it.next()) {
            const int kcb = it.kc_begin(), kce = it.kc_end();
            for (int kc = kcb; kc < kce; ++kc) {
                umma::mbar_wait(&full_bar[stage], phase);
                auto convert = [&](uint8_t* hi_slot, int slot_bytes, bool is_a) {
                    float4* xh = reinterpret_cast<float4*>(hi_slot);
                    float4* xl = reinterpret_cast<float4*>(hi_slot + slot_bytes);
#pragma unroll 4
                    for (int j = ct; j < slot_bytes / 16; j += 32 * UG_CONV_WARPS) {
                        float4 x = xh[j];
                        if constexpr (epi_transforms_a<Epi>::value) {
                            // element-wise map applied to the A operand on its way into the tensor core (K4b: the RBF kernel
                            // exp(-D2 / 2bw) is never materialised -- the GEMM reads D2 and multiplies by its exponential)
                            if (is_a) { x.x = Epi::transform_a(a_ctx, x.x); x.y = Epi::transform_a(a_ctx, x.y);
                                        x.z = Epi::transform_a(a_ctx, x.z); x.w = Epi::transform_a(a_ctx, x.w); }
                        }
                        float4 h, l;
                        umma::split_tf32(x.x, h.x, l.x); umma::split_tf32(x.y, h.y, l.y);
                        umma::split_tf32(x.z, h.z, l.z); umma::split_tf32(x.w, h.w, l.w);
                        xh[j] = h;
                        xl[j] = l;
                    }
                };
                uint8_t* st = smem + stage * SM::STAGE_BYTES;
                if (SPLIT_A) convert(st, SM::A_BYTES, true);
                if (SPLIT_B) convert(st + 2 * SM::A_BYTES, SM::B_BYTES, false);
                umma::fence_proxy_async();        // generic-proxy writes -> visible to the tensor core's async-proxy reads
                __syncwarp();
                if (lane == 0) umma::mbar_arrive(&conv_bar[stage]);
                if (++stage == UG_STAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else {
        // ===================== epilogue warps =====================
        const int ew = warp - 2;
        const int q = warp & 3;                   // TMEM lane quarter this warp may access (warp id % 4)
        const int hf = ew >> 2;                   // column block (half / quarter of the tile)
        const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16) + hf * CPT;
        uint32_t blk = 0;
        for (UnitIter it(m_tiles, n_tiles, k_chunks, mode, split_T, full_units); it.valid(); it.next()) {
            float r[CPT];
#pragma unroll
            for (int i = 0; i < CPT; ++i) r[i] = 0.f;
            const int kcb = it.kc_begin(), kce = it.kc_end();
            for (int kc0 = kcb; kc0 < kce; kc0 += drain_chunks, ++blk) {
                const uint32_t buf = blk & 1, use = (blk >> 1) & 1;
                umma::mbar_wait(&acc_full[buf], use);
                umma::tc_fence_after();
                const uint32_t t0 = t_lane + buf * UG_BUF_COLS;
                constexpr int C32 = EW == 16 ? 0 : CPT / 32 * 32;     // 16 warps: 16-column pieces only (register budget 112)
#pragma unroll
                for (int c = 0; c + 32 <= C32; c += 32) {
                    float v[32];
                    umma::tmem_ld_32x32(t0 + c, v);
                    umma::tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 32; ++i) r[c + i] += v[i];
                }
#pragma unroll
                for (int c = C32; c + 16 <= CPT; c += 16) {
                    float v[16];
                    umma::tmem_ld_32x16(t0 + c, v);
                    umma::tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 16; ++i) r[c + i] += v[i];
                }
                if (CPT % 16 == 8) {
                    float v[8];
                    umma::tmem_ld_32x8(t0 + (CPT / 16) * 16, v);
                    umma::tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 8; ++i) r[(CPT / 16) * 16 + i] += v[i];
                }
                umma::tc_fence_before();
                __syncwarp();
                if (lane == 0) umma::mbar_arrive(&acc_empty[buf]);
            }
            Epi::finish(ep, r, it.mt() * UG_BM + q * 32 + lane, it.nt() * (EW / 4) + hf, it.in_tail(), it.slice());
        }
    }
    umma::tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        umma::tc_fence_after();
        umma::tmem_dealloc(tmem_base, TMEM_COLS);
    }
}

// ------------------------------------------------------------------------------------------------
// epilogue policy: strided store.  An epilogue thread owns one tile row and one half of the tile's
// columns = one "block" of CPT columns (for K3: one MC sample):
//     out[blk * blk_stride + row * row_stride + col * col_stride]      col < valid(blk), row < rows
// row_stride == 1 gives the transposed (coalesced across the warp) store both K3 GEMMs use.
// ------------------------------------------------------------------------------------------------
// epilogue policy for tile-shape measurements: drains the accumulators and writes nothing
struct EpiNull {
    struct Params { float* out; };
    template <int CPT>
    static __device__ __forceinline__ void finish(const Params& p, float (&r)[CPT], int row, int blk, bool, int) {
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < CPT; ++i) s += r[i];
        if (s == 1.2345e-30f) p.out[0] = s;      // keeps the drain alive
    }
};

// power of two s with m * s in [2^13, 2^14)  (m > 0; 1 for m == 0 or non-finite): the operand scaling of the fp16 kind
__device__ __forceinline__ float p2_scale(float m) {
    if (!(m > 0.f) || !(m < 3.0e38f)) return 1.f;
    int e = (int)((__float_as_uint(m) >> 23) & 0xffu) - 127;
    e = max(-100, min(100, e));
    return __uint_as_float((uint32_t)(127 + 13 - e) << 23);
}

struct EpiStore {
    struct Params {
        float* out; int rows; int64_t row_stride, col_stride, blk_stride;
        int blk_valid;      // valid columns per block ...
        int col_limit;      // ... or, if > 0, total valid columns counted across consecutive blocks
        int total_blks;
        // fp16 kind: the operands were scaled by p2_scale(*bound_a) and p2_scale(bound_b_mult * *bound_b) (device scalars)
        const float* bound_a = nullptr; const float* bound_b = nullptr; float bound_b_mult = 1.f;
    };
    template <int CPT>
    static __device__ __forceinline__ void finish(const Params& p, float (&r)[CPT], int row, int blk, bool accumulate, int /*slice*/) {
        if (row >= p.rows || blk >= p.total_blks) return;
        if (p.bound_a) {
            const float inv = 1.f / (p2_scale(*p.bound_a) * p2_scale(p.bound_b_mult * *p.bound_b));
#pragma unroll
            for (int i = 0; i < CPT; ++i) r[i] *= inv;
        }
        int valid = p.blk_valid;
        if (p.col_limit > 0) valid = min(CPT, p.col_limit - blk * CPT);
        float* o = p.out + (int64_t)blk * p.blk_stride + (int64_t)row * p.row_stride;
        if (accumulate) {          // K-split tail unit: partial sums into the caller-zeroed block
#pragma unroll
            for (int i = 0; i < CPT; ++i)
                if (i < valid) atomicAdd(&o[(int64_t)i * p.col_stride], r[i]);
        } else {
#pragma unroll
            for (int i = 0; i < CPT; ++i)
                if (i < valid) o[(int64_t)i * p.col_stride] = r[i];
        }
    }
};

// ------------------------------------------------------------------------------------------------
// epilogue policy: K-slice accumulation without atomics.  Unit (row tile, column half) of K-slice j owns
//     out[j * slice_stride + row * ld + col]   and adds its result to what is there (stream-ordered launches of the
// same shape accumulate chunk after chunk; a final pass sums the slices).  Deterministic, unlike atomics.
// ------------------------------------------------------------------------------------------------
struct EpiAccum {
    struct Params {
        float* out; int rows, cols; int64_t ld, slice_stride;
    };
    template <int CPT>
    static __device__ __forceinline__ void finish(const Params& p, float (&r)[CPT], int row, int blk, bool, int slice) {
        if (row >= p.rows) return;
        float* o = p.out + (int64_t)slice * p.slice_stride + (int64_t)row * p.ld + (int64_t)blk * CPT;
        const int valid = min(CPT, p.cols - blk * CPT);
        if (valid == CPT && ((reinterpret_cast<uintptr_t>(o) & 15) == 0)) {
#pragma unroll
            for (int i = 0; i < CPT; i += 4) {
                float4 v = *reinterpret_cast<float4*>(o + i);
                v.x += r[i]; v.y += r[i + 1]; v.z += r[i + 2]; v.w += r[i + 3];
                *reinterpret_cast<float4*>(o + i) = v;
            }
        } else {
#pragma unroll
            for (int i = 0; i < CPT; ++i)
                if (i < valid) o[i] += r[i];
        }
    }
};

// ------------------------------------------------------------------------------------------------
// epilogue policy: Bernoulli / Binomial(1) likelihood fused behind the logits GEMM (K2):
//   D[row n, col s] = logit;  ll += y_n l - log(1 + e^l);  d = y_n - sigmoid(l)
//   d is written as plain fp32 and TRANSPOSED: dT[s * ld + n]  (the K-major A operand of the gradient GEMM, which splits it
//   on the fly (SPLIT & 1) -- half the bytes through HBM; coalesced across the warp's 32 rows).  log1p(e^-|l|) is evaluated as log(1 + e): its absolute error (< 6e-8)
//   is far below the fp32 resolution of the terms it is added to.
// ------------------------------------------------------------------------------------------------
struct EpiBernoulli {
    struct Params {
        const float* y; float* dT; int rows, cols; int64_t ld; double* loss; float neg_inv_S;
    };
    // one element: log-likelihood term and the gradient d = y - sigmoid(l).  MUFU ex2 / rcp / lg2 (absolute errors
    // ~1e-7, far inside the parity budget), no slow-path calls: the epilogue warps are the pace-setter of this GEMM (K = F
    // is short), so every instruction here is on the critical path (profiles/r1g_ncu_full_logreg_summary.txt).
    static __device__ __forceinline__ float element(float l, float yv, float& d) {
        float e, inv, lg;
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-1.4426950408889634f * fabsf(l)));
        const float ope = 1.f + e;
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(inv) : "f"(ope));
        asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(ope));
        const float sig = l >= 0.f ? inv : e * inv;
        d = yv - sig;
        return __fmaf_rn(yv, l, -__fmaf_rn(lg, 0.6931471805599453f, fmaxf(l, 0.f)));
    }
    template <int CPT>
    static __device__ __forceinline__ void finish(const Params& p, float (&r)[CPT], int row, int blk, bool, int) {
        const bool row_ok = row < p.rows;
        const float yv = row_ok ? p.y[row] : 0.f;
        const int valid = row_ok ? min(CPT, p.cols - blk * CPT) : 0;
        float ll = 0.f;
        const int64_t ld = p.ld;
        float* o = p.dT + (int64_t)blk * CPT * ld + row;
#pragma unroll          // full unroll: r[] must stay in registers (a partial unroll indexes it dynamically -> local memory)
        for (int i = 0; i < CPT; ++i) {
            if (i < valid) {
                float d;
                ll += element(r[i], yv, d);
                o[0] = d;
            }
            o += ld;
        }
        double tot = (double)ll;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, o);
        if ((threadIdx.x & 31) == 0 && tot != 0.0) atomicAdd(p.loss, tot * (double)p.neg_inv_S);
    }
};

int launch_split_tf32(const float* src, int64_t lds, int rows, int cols, float* hi, float* lo, int64_t ldd, float* thi,
                      float* tlo, int64_t ldt, cudaStream_t stream);
int launch_transpose_f32(const float* src, int64_t lds, int rows, int cols, float* dst, int64_t ldt, cudaStream_t stream);

// Work split of mode 0 on `sms` CTAs: grid size, and -- when the last round-robin round would be at most half full --
// the K-split of the tail units (see UnitIter).  first_split_ntile = first n-tile whose output blocks receive atomic
// partial sums and must be ZEROED by the caller before the launch (-1: no split).
struct UmmaSplitPlan {
    int grid, split_T, full_units, first_split_ntile;
};
template <int BN, int BK>
inline UmmaSplitPlan umma_plan(int M, int N, int K, int sms, bool allow_split) {
    const int m_tiles = (M + UG_BM - 1) / UG_BM, n_tiles = (N + BN - 1) / BN, k_chunks = (K + BK - 1) / BK;
    const int U = m_tiles * n_tiles;
    UmmaSplitPlan p;
    p.grid = U < sms ? U : sms;
    p.split_T = 0; p.full_units = U; p.first_split_ntile = -1;
    const int T = U % p.grid;
    if (allow_split && U > p.grid && T > 0 && 2 * T <= p.grid && k_chunks >= 2 * (p.grid / T)) {
        p.split_T = T;
        p.full_units = U - T;
        p.first_split_ntile = p.full_units / m_tiles;
    } else if (allow_split && 2 * U <= sms && k_chunks >= 2 * (sms / U)) {
        p.grid = sms / U * U;           // every unit is K-split over sms/U CTAs
        p.split_T = U;
        p.full_units = 0;
        p.first_split_ntile = 0;
    }
    return p;
}

// A (hi/lo) [M][K] pitch lda, B (hi/lo) [N][K] pitch ldb; mode 0: units n-major round-robin over CTAs,
// mode 1: every CTA keeps one m-tile and strides over n-tiles.  allow_split: the caller has zeroed the output blocks of
// n-tiles >= umma_plan(...).first_split_ntile (mode 0 only).
template <int BN, int BK, class Epi, int EW = UG_EPI_WARPS, int SPLIT = 0, int CW = 4, int KIND = 0>
inline int launch_umma_nt_kind(const void* Ah, const void* Al, int M, int64_t lda, const void* Bh, const void* Bl, int N,
                               int64_t ldb, int K, int mode, int drain_chunks, const typename Epi::Params& ep,
                               cudaStream_t stream, bool allow_split = false) {
    constexpr int KE = KIND == 0 ? 1 : 2;
    CUtensorMap tAh, tAl, tBh, tBl;
    auto mk = [](CUtensorMap* t, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows) {
        return KIND == 0 ? make_tmap_2d_f32(t, static_cast<const float*>(base), rows, cols, ld, box_rows, BK)
                         : make_tmap_2d_f16(t, base, rows, cols, ld, box_rows, BK * 2);
    };
    if (int e = mk(&tAh, Ah, M, K, lda, UG_BM)) return e;
    if (int e = mk(&tAl, (SPLIT & 1) ? Ah : Al, M, K, lda, UG_BM)) return e;      // SPLIT & 1: unused
    if (int e = mk(&tBh, Bh, N, K, ldb, BN)) return e;
    if (int e = mk(&tBl, (SPLIT & 2) ? Bh : Bl, N, K, ldb, BN)) return e;        // SPLIT & 2: unused
    const int m_tiles = (M + UG_BM - 1) / UG_BM, n_tiles = (N + BN - 1) / BN, k_chunks = (K + BK * KE - 1) / (BK * KE);
    drain_chunks = drain_chunks * 32 / BK;        // `drain_chunks` is given in units of 32 words of K
    const int sms = device_sm_count();
    int grid, split_T = 0, full_units = m_tiles * n_tiles;
    if (mode == 0 || mode == 2) {
        const UmmaSplitPlan pl = umma_plan<BN, BK * KE>(M, N, K, sms, allow_split && mode == 0);
        grid = pl.grid; split_T = pl.split_T; full_units = pl.full_units;
    } else {
        int G = sms / m_tiles;
        if (G < 1) G = 1;
        if (G > n_tiles) G = n_tiles;
        grid = G * m_tiles;
    }
    if (drain_chunks < 1) drain_chunks = 2 * 32 / BK;
    auto kern = umma_nt_3xtf32_kernel<BN, BK, Epi, EW, SPLIT, CW, KIND>;
    const int smem = UmmaSmem<BN, BK>::TOTAL;
    BRN_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    kern<<<grid, 64 + 32 * EW + (SPLIT ? 32 * CW : 0), smem, stream>>>(tAh, tAl, tBh, tBl, m_tiles, n_tiles, k_chunks, drain_chunks, mode,
                                                         split_T, full_units, ep);
    BRN_LAUNCH_OK("umma_nt_3xtf32_kernel");
    return 0;
}

template <int BN, int BK, class Epi, int EW = UG_EPI_WARPS, int SPLIT = 0, int CW = 4>
inline int launch_umma_nt(const float* Ah, const float* Al, int M, int64_t lda, const float* Bh, const float* Bl, int N,
                          int64_t ldb, int K, int mode, int drain_chunks, const typename Epi::Params& ep,
                          cudaStream_t stream, bool allow_split = false) {
    return launch_umma_nt_kind<BN, BK, Epi, EW, SPLIT, CW, 0>(Ah, Al, M, lda, Bh, Bl, N, ldb, K, mode, drain_chunks, ep, stream,
                                                              allow_split);
}

// D [M][N] = sum_k A[k][m] B[k][n]: A [K][M] pitch lda and B [K][N] pitch ldb, both plain fp32 row-major (split into TF32 pairs
// by the converter warps: SPLIT = 3), read MN-major.  mode / allow_split as launch_umma_nt.
template <int BN, int BK, class Epi, int EW = UG_EPI_WARPS, int CW = 4>
inline int launch_umma_tn_plain(const float* A, int M, int64_t lda, const float* B, int N, int64_t ldb, int K, int mode,
                                int drain_chunks, const typename Epi::Params& ep, cudaStream_t stream, bool allow_split = false) {
    CUtensorMap tA, tB;
    if (int e = make_tmap_2d_f32(&tA, A, K, M, lda, BK, 32, true)) return e;
    if (int e = make_tmap_2d_f32(&tB, B, K, N, ldb, BK, 32, true)) return e;
    const int m_tiles = (M + UG_BM - 1) / UG_BM, n_tiles = (N + BN - 1) / BN, k_chunks = (K + BK - 1) / BK;
    drain_chunks = drain_chunks * 32 / BK;
    const int sms = device_sm_count();
    const UmmaSplitPlan pl = umma_plan<BN, BK>(M, N, K, sms, allow_split && mode == 0);
    if (drain_chunks < 1) drain_chunks = 2 * 32 / BK;
    auto kern = umma_nt_3xtf32_kernel<BN, BK, Epi, EW, 3, CW, 0, 1>;
    const int smem = UmmaSmem<BN, BK>::TOTAL;
    BRN_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    kern<<<pl.grid, 64 + 32 * EW + 32 * CW, smem, stream>>>(tA, tA, tB, tB, m_tiles, n_tiles, k_chunks, drain_chunks, mode, pl.split_T,
                                                          pl.full_units, ep);
    BRN_LAUNCH_OK("umma_nt_3xtf32_kernel (MN-major)");
    return 0;
}

}  // namespace brn
