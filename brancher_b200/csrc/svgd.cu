// K4: Stein variational gradient descent direction -- pairwise RBF kernel + "repulsive" term as a tiled n^2 kernel.
// See include/brancher_cuda.h (brn_svgd_direction) for the contract and the reference lines replaced
// (brancher/inference.py:301-324, four nested Python loops over numpy scalars).
//
//   D2_ij = ||theta_i - theta_j||^2                                    svgd_d2_kernel     (n^2 d, direct differences)
//   bw    = 2 median_{i != j}(sqrt D2_ij)^2 / ln n                     svgd_select_*      (exact radix select)
//   out_i = sum_j K_ij (g_j - theta_j / bw) + theta_i rowsum_i(K) / bw svgd_update_kernel (K_ij = exp(-D2_ij / 2bw))
//
// The median is EXACT (np.median semantics: mean of the two middle order statistics): because D2 is symmetric the
// multiset {D2_ij : i != j} is the multiset {D2_ij : i < j} with every element doubled, which has the same median,
// so the select runs over the m = n(n-1)/2 upper-triangle values.  Non-negative floats order like their bit
// patterns: three histogram passes (12 + 12 + 8 bits) pin the k-th smallest value, one more pass finds its successor.
#include "umma_gemm.cuh"
#include <stdlib.h>
#include <cstddef>

namespace brn {

constexpr int SV_T = 64;        // D2 tile edge
constexpr int SV_KC = 32;       // feature chunk

// D2[i][j] for a 64x64 tile; 256 threads, 4x4 outputs per thread.
__global__ void __launch_bounds__(256) svgd_d2_kernel(const float* __restrict__ theta, int n, int d, float* __restrict__ D2) {
    __shared__ float As[SV_KC][SV_T + 4], Bs[SV_KC][SV_T + 4];      // [k][row]
    const int i0 = blockIdx.y * SV_T, j0 = blockIdx.x * SV_T;
    const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
    float acc[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;
    for (int k0 = 0; k0 < d; k0 += SV_KC) {
        __syncthreads();
        for (int idx = t; idx < SV_T * SV_KC; idx += 256) {
            const int row = idx / SV_KC, k = idx - row * SV_KC;
            const bool kok = k0 + k < d;
            As[k][row] = (kok && i0 + row < n) ? theta[(int64_t)(i0 + row) * d + k0 + k] : 0.f;
            Bs[k][row] = (kok && j0 + row < n) ? theta[(int64_t)(j0 + row) * d + k0 + k] : 0.f;
        }
        __syncthreads();
#pragma unroll 8
        for (int k = 0; k < SV_KC; ++k) {
            const float4 a4 = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
            const float4 b4 = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
            const float av[4] = {a4.x, a4.y, a4.z, a4.w}, bv[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    const float df = av[a] - bv[b];
                    acc[a][b] = __fmaf_rn(df, df, acc[a][b]);
                }
        }
    }
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        const int i = i0 + ty * 4 + a;
        if (i >= n) continue;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const int j = j0 + tx * 4 + b;
            if (j < n) D2[(int64_t)i * n + j] = acc[a][b];
        }
    }
}

struct SelectState {
    unsigned long long rank;     // remaining 0-based rank inside the current prefix bucket
    unsigned long long cnt_le;   // pass 4: #{v <= selected}
    uint32_t prefix;             // high bits fixed so far (value of the k1-th smallest after the 3rd scan)
    uint32_t next;               // pass 4: min{v > selected} (bit pattern)
};

// histogram of bits [shift, shift+nbits) over the upper-triangle elements (j > i) of rows [row0, row0 + rows) whose higher bits
// equal state->prefix.  D2 points at row `row0` (row pitch n): the whole matrix (row0 = 0, rows = n) or one rank's row shard,
// whose partial histograms add up to the full one because every row belongs to exactly one rank.
__global__ void __launch_bounds__(256) svgd_select_hist_kernel(const float* __restrict__ D2, int n, int row0, int rows, int shift,
                                                               int nbits, int first, const SelectState* __restrict__ st,
                                                               unsigned int* __restrict__ hist) {
    extern __shared__ unsigned int sh[];
    const int nb = 1 << nbits;
    for (int b = threadIdx.x; b < nb; b += blockDim.x) sh[b] = 0u;
    __syncthreads();
    const uint32_t prefix = first ? 0u : st->prefix;
    const int hshift = shift + nbits;
    // rows are dealt round-robin to the CTAs; a row's upper-triangle part (j > i) is read coalesced -- the lower triangle is
    // never touched and no index division is needed
    // (local rows q and rows-1-q are handled together: their upper-triangle lengths add up to a constant, which balances the CTAs)
    for (int q = blockIdx.x; 2 * q < rows; q += gridDim.x)
    for (int h = 0; h < 2; ++h) {
        const int li = h == 0 ? q : rows - 1 - q;
        if (h == 1 && li <= q) continue;
        const int i = row0 + li;
        const float* row = D2 + (int64_t)li * n;
        for (int jb = i + 1; jb < n; jb += blockDim.x) {      // warp-uniform trip count: the ballot below needs all lanes
            const int j = jb + threadIdx.x;
            bool take = false;
            uint32_t bin = 0;
            if (j < n) {
                const uint32_t v = __float_as_uint(row[j]);
                if (first || (hshift < 32 && (v >> hshift) == (prefix >> hshift))) {
                    take = true;
                    bin = (v >> shift) & (uint32_t)(nb - 1);
                }
            }
            // warp-aggregated shared atomics: distances concentrate in a handful of bins
            const unsigned active = __ballot_sync(0xffffffffu, take);
            if (take) {
                const unsigned peers = __match_any_sync(active, bin);
                if ((int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&sh[bin], (unsigned)__popc(peers));
            }
        }
    }
    __syncthreads();
    for (int b = threadIdx.x; b < nb; b += blockDim.x)
        if (sh[b]) atomicAdd(&hist[b], sh[b]);
}

// one block of 1024 threads: find the bin holding the wanted rank with a block-wide prefix scan of the histogram (thread t owns
// `per` consecutive bins), extend the prefix, clear the histogram.  (The first version walked the 4096 bins with ONE thread:
// 4096 dependent L2 loads = 112 us per level, 14 % of the whole SVGD step -- profiles/r1g_launches_svgd_summary.txt.)
constexpr int SCAN_THREADS = 1024;
__global__ void __launch_bounds__(SCAN_THREADS) svgd_select_scan_kernel(int shift, int nbits, int first, unsigned long long k,
                                                                        SelectState* st, unsigned int* hist) {
    __shared__ unsigned long long warp_tot[SCAN_THREADS / 32];
    __shared__ unsigned long long s_rank;
    __shared__ int s_bin;
    const int nb = 1 << nbits, per = (nb + SCAN_THREADS - 1) / SCAN_THREADS;      // per <= 4 (nbits <= 12)
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    const unsigned long long rank0 = first ? k : st->rank;
    const uint32_t prefix = first ? 0u : st->prefix;
    unsigned int c[4] = {0u, 0u, 0u, 0u};
    unsigned long long loc = 0ull;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int b = t * per + j;
        if (j < per && b < nb) c[j] = hist[b];
        loc += c[j];
    }
    unsigned long long inc = loc;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long up = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += up;
    }
    if (lane == 31) warp_tot[w] = inc;
    if (t == 0) { s_bin = -1; s_rank = 0ull; }
    __syncthreads();
    if (w == 0) {
        unsigned long long x = warp_tot[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long up = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += up;
        }
        warp_tot[lane] = x;          // inclusive prefix over warps
    }
    __syncthreads();
    const unsigned long long excl = inc - loc + (w > 0 ? warp_tot[w - 1] : 0ull);
    if (rank0 >= excl && rank0 < excl + loc) {             // exactly one thread (bins are disjoint, counts are non-negative)
        unsigned long long r = rank0 - excl;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (j < per && s_bin < 0) {
                if (r < c[j]) { s_bin = t * per + j; s_rank = r; }
                else r -= c[j];
            }
        }
    }
    __syncthreads();
    if (t == 0) {
        int b = s_bin;
        unsigned long long rank = s_rank;
        if (b < 0) {                 // rank beyond the histogram total (cannot happen for a consistent state): last bin, as the
            b = nb - 1;              // serial walk did
            rank = rank0 - (warp_tot[SCAN_THREADS / 32 - 1] - hist[nb - 1]);
        }
        st->rank = rank;
        st->prefix = prefix | ((uint32_t)b << shift);
        st->cnt_le = 0ull;
        st->next = 0x7f800000u;       // +inf
    }
    __syncthreads();
    for (int b = t; b < nb; b += SCAN_THREADS) hist[b] = 0u;
}

// pass 4: count of values <= selected and the smallest value above it (same row range convention as the histogram)
__global__ void __launch_bounds__(256) svgd_select_succ_kernel(const float* __restrict__ D2, int n, int row0, int rows, SelectState* st) {
    const uint32_t sel = st->prefix;
    unsigned long long cnt = 0ull;
    uint32_t nxt = 0x7f800000u;
    for (int q = blockIdx.x; 2 * q < rows; q += gridDim.x)
    for (int h = 0; h < 2; ++h) {
        const int li = h == 0 ? q : rows - 1 - q;
        if (h == 1 && li <= q) continue;
        const int i = row0 + li;
        const float* row = D2 + (int64_t)li * n;
        for (int j = i + 1 + threadIdx.x; j < n; j += blockDim.x) {
            const uint32_t v = __float_as_uint(row[j]);
            if (v <= sel) ++cnt;
            else nxt = min(nxt, v);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
        nxt = min(nxt, __shfl_xor_sync(0xffffffffu, nxt, o));
    }
    if ((threadIdx.x & 31) == 0) {
        if (cnt) atomicAdd(&st->cnt_le, cnt);
        atomicMin(&st->next, nxt);
    }
}

// bw = 2 * median(dist)^2 / ln n with median = (sqrt(v_k1) + sqrt(v_k2)) / 2   (np.median of float32 distances)
__global__ void svgd_bandwidth_kernel(const SelectState* st, unsigned long long k2, int n, float* bw) {
    if (threadIdx.x == 0) {
        const float v1 = __uint_as_float(st->prefix);
        const float v2 = st->cnt_le >= k2 + 1ull ? v1 : __uint_as_float(st->next);
        const float med = 0.5f * (sqrtf(v1) + sqrtf(v2));
        *bw = (float)(2.0 * (double)(med * med) / log((double)n));
    }
}

// out[i, :] (+)= sum_j K_ij (g_j - theta_j / bw) + theta_i rowsum_i(K) / bw over this CTA's j range.
// CTA: 32 rows x 128 columns, 128 threads (4 rows x 8 columns each), j tiles of 32; grid = (row tiles, d chunks, j splits).
constexpr int SU_TI = 32, SU_TJ = 32, SU_TD = 128;

__global__ void __launch_bounds__(128)
svgd_update_kernel(const float* __restrict__ theta, const float* __restrict__ grad, const float* __restrict__ D2, int n, int d,
                   int row0, int rows, const float* __restrict__ bw_ptr, float* __restrict__ out, int j_per_split) {
    __shared__ __align__(16) float Ks[SU_TJ][SU_TI + 4];     // [jj][ii]
    __shared__ __align__(16) float Vs[SU_TJ][SU_TD + 4];     // [jj][col]
    __shared__ float rs_s[SU_TI];
    const int t = threadIdx.x, tx = t & 15, ty = t >> 4;     // ty: 0..7 -> rows ty*4.., tx: cols tx*4.. and 64+tx*4..
    const int i0 = row0 + blockIdx.x * SU_TI, c0 = blockIdx.y * SU_TD;
    const int jbeg = blockIdx.z * j_per_split, jend = min(n, jbeg + j_per_split);
    const int iend = row0 + rows;
    const float bw = *bw_ptr, inv_bw = 1.0f / bw, nh = -0.5f / bw;
    float acc[4][8];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 8; ++b) acc[a][b] = 0.f;
    float rs[4] = {0.f, 0.f, 0.f, 0.f};

    for (int j0 = jbeg; j0 < jend; j0 += SU_TJ) {
        __syncthreads();
        for (int idx = t; idx < SU_TI * SU_TJ; idx += 128) {
            const int ii = idx >> 5, jj = idx & 31;
            float kv = 0.f;
            if (i0 + ii < iend && j0 + jj < jend) kv = expf(nh * D2[(int64_t)(i0 + ii) * n + j0 + jj]);
            Ks[jj][ii] = kv;
        }
        for (int idx = t; idx < SU_TJ * (SU_TD / 4); idx += 128) {
            const int jj = idx >> 5, c4 = (idx & 31) * 4;
            float v[4] = {0.f, 0.f, 0.f, 0.f};
            if (j0 + jj < jend) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int c = c0 + c4 + q;
                    if (c < d) {
                        const int64_t o = (int64_t)(j0 + jj) * d + c;
                        v[q] = __fmaf_rn(-theta[o], inv_bw, grad[o]);
                    }
                }
            }
            *reinterpret_cast<float4*>(&Vs[jj][c4]) = make_float4(v[0], v[1], v[2], v[3]);
        }
        __syncthreads();
#pragma unroll 8
        for (int jj = 0; jj < SU_TJ; ++jj) {
            const float4 a4 = *reinterpret_cast<const float4*>(&Ks[jj][ty * 4]);
            const float4 b0 = *reinterpret_cast<const float4*>(&Vs[jj][tx * 4]);
            const float4 b1 = *reinterpret_cast<const float4*>(&Vs[jj][64 + tx * 4]);
            const float av[4] = {a4.x, a4.y, a4.z, a4.w};
            const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int a = 0; a < 4; ++a) {
                if (tx == 0) rs[a] += av[a];
#pragma unroll
                for (int b = 0; b < 8; ++b) acc[a][b] = __fmaf_rn(av[a], bv[b], acc[a][b]);
            }
        }
    }
    if (tx == 0) {
#pragma unroll
        for (int a = 0; a < 4; ++a) rs_s[ty * 4 + a] = rs[a];
    }
    __syncthreads();
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        const int i = i0 + ty * 4 + a;
        if (i >= iend) continue;
        const float w = rs_s[ty * 4 + a] * inv_bw;
#pragma unroll
        for (int b = 0; b < 8; ++b) {
            const int c = c0 + (b < 4 ? tx * 4 + b : 64 + tx * 4 + (b - 4));
            if (c >= d) continue;
            const float v = __fmaf_rn(theta[(int64_t)i * d + c], w, acc[a][b]);
            float* o = out + (int64_t)(i - row0) * d + c;
            if (gridDim.z == 1) *o = v;
            else atomicAdd(o, v);
        }
    }
}


// ---------------------------------------------------------------------------------------------------
// tensor-core variant of the two contractions (tcgen05, 3xTF32):
//   D2 = |a|^2 + |b|^2 - 2 a.b   -- theta . theta^T through the GEMM, norms and clamp in its epilogue (EpiD2)
//   out = K . [g - theta / bw | 1] -- the GEMM reads D2 itself; its converter warps turn every element into
//         exp(-D2 / 2bw) on its way into the tensor core (TRANSFORMS_A), so the kernel matrix K is never materialised;
//         the appended column of ones delivers rowsum(K) for the attractive term (EpiSvgdOut).
// ---------------------------------------------------------------------------------------------------
struct EpiD2 {
    struct Params { const float* sq; float* D2; int rows, n; int row0; };
    template <int CPT>
    static __device__ __forceinline__ void finish(const Params& p, float (&r)[CPT], int row, int blk, bool, int) {
        if (row >= p.rows) return;
        const int gi = p.row0 + row, c0 = blk * CPT;
        const float si = p.sq[gi];
        float* o = p.D2 + (int64_t)row * p.n + c0;
#pragma unroll
        for (int i = 0; i < CPT; i += 4) {
            float v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int j = c0 + i + u;
                float x = 0.f;
                if (j < p.n && j != gi) x = fmaxf(__fmaf_rn(-2.f, r[i + u], si + p.sq[j]), 0.f);
                v[u] = x;
            }
            if (c0 + i + 3 < p.n && (p.n & 3) == 0) *reinterpret_cast<float4*>(o + i) = make_float4(v[0], v[1], v[2], v[3]);
            else {
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (c0 + i + u < p.n) o[i + u] = v[u];
            }
        }
    }
};

struct EpiSvgdOut {
    static constexpr bool TRANSFORMS_A = true;
    struct Params { float* out; const float* theta; const float* bw; int rows, d, row0; };
    static __device__ __forceinline__ float transform_a_context(const Params& p) { return -0.5f / *p.bw * 1.4426950408889634f; }
    static __device__ __forceinline__ float transform_a(float ctx, float x) {
        float e;
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * ctx));
        return e;
    }
    // one thread = one particle row and all d + 1 accumulator columns (column d = rowsum of K); K-split slices add up
    template <int CPT>
    static __device__ __forceinline__ void finish(const Params& p, float (&r)[CPT], int row, int blk, bool, int) {
        if (row >= p.rows || blk != 0) return;
        float rowsum = 0.f;                                            // column d (d < CPT by construction); static indexing only
#pragma unroll
        for (int c = 0; c < CPT; ++c)
            if (c == p.d) rowsum = r[c];
        const float w = rowsum / *p.bw;
        const float* th = p.theta + (int64_t)(p.row0 + row) * p.d;
        float* o = p.out + (int64_t)row * p.d;
#pragma unroll
        for (int c = 0; c < CPT; ++c)
            if (c < p.d) atomicAdd(o + c, __fmaf_rn(th[c], w, r[c]));
    }
};

// sq[i] = |theta_i|^2 and the TF32 (hi, lo) pair of theta [n][ld]
__global__ void __launch_bounds__(128) svgd_prep_theta_kernel(const float* __restrict__ theta, int n, int d, int64_t ld,
                                                              float* __restrict__ hi, float* __restrict__ lo, float* __restrict__ sq) {
    const int i = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (i >= n) return;
    float acc = 0.f;
    for (int c = lane; c < d; c += 32) {
        const float x = theta[(int64_t)i * d + c];
        float h, l;
        umma::split_tf32(x, h, l);
        hi[(int64_t)i * ld + c] = h;
        lo[(int64_t)i * ld + c] = l;
        acc = __fmaf_rn(x, x, acc);
    }
    acc = warp_sum(acc);
    if (lane == 0) sq[i] = acc;
}

// Vt[c][j] = g[j][c] - theta[j][c] / bw (c < d), Vt[d][j] = 1: the K-major B operand [d + 1][ldn] as a TF32 (hi, lo) pair
__global__ void __launch_bounds__(256) svgd_prep_v_kernel(const float* __restrict__ theta, const float* __restrict__ grad, int n,
                                                          int d, const float* __restrict__ bw, float* __restrict__ hi,
                                                          float* __restrict__ lo, int64_t ldn) {
    __shared__ float t[32][33];
    const float inv_bw = 1.0f / *bw;
    const int j0 = blockIdx.x * 32, c0 = blockIdx.y * 32, tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int r = ty; r < 32; r += 8) {
        const int j = j0 + r, c = c0 + tx;
        float v = 0.f;
        if (j < n) {
            if (c < d) v = __fmaf_rn(-theta[(int64_t)j * d + c], inv_bw, grad[(int64_t)j * d + c]);
            else if (c == d) v = 1.f;
        }
        t[r][tx] = v;
    }
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {
        const int c = c0 + r, j = j0 + tx;
        if (c <= d && j < n) {
            float h, l;
            umma::split_tf32(t[tx][r], h, l);
            hi[(int64_t)c * ldn + j] = h;
            lo[(int64_t)c * ldn + j] = l;
        }
    }
}

constexpr int SVGD_TC_BN = 144;        // update GEMM N tile: d + 1 <= 144

struct SvgdWorkspace {
    float* D2;
    unsigned int* hist;
    SelectState* st;
    float *th_hi, *th_lo, *sq, *vt_hi, *vt_lo;
    int64_t ldd, ldn;
    size_t bytes;
    size_t hist_off, st_off;
    // d2_rows: rows of D2 kept (n for the replicated evaluation, the rank's shard for the sharded one)
    SvgdWorkspace(void* base, int n, int d, int d2_rows = -1) {
        if (d2_rows < 0) d2_rows = n;
        WorkspaceCarver take(base);
        D2 = take((size_t)(d2_rows > 0 ? d2_rows : 1) * n);
        hist_off = take.off;
        hist = reinterpret_cast<unsigned int*>(take.bytes(sizeof(unsigned int) * 4096));
        st_off = take.off;
        st = reinterpret_cast<SelectState*>(take.bytes(sizeof(SelectState)));
        // tensor-core variant: theta (hi, lo) [n][ldd], |theta|^2 [n], V^T (hi, lo) [d + 1][ldn]
        ldd = (d + 3) / 4 * 4;
        ldn = (n + 3) / 4 * 4;
        th_hi = take((size_t)n * ldd);
        th_lo = take((size_t)n * ldd);
        sq = take((size_t)n);
        vt_hi = take((size_t)(d + 1) * ldn);
        vt_lo = take((size_t)(d + 1) * ldn);
        bytes = take.off;
    }
};

}  // namespace brn

using namespace brn;

extern "C" size_t brn_svgd_workspace_bytes(int n, int d) {
    if (n <= 0 || d <= 0) return 0;
    return SvgdWorkspace(nullptr, n, d).bytes;
}

extern "C" int brn_svgd_direction(const float* theta, const float* grad, int n, int d, int row0, int rows,
                                  int update_bandwidth, float* bandwidth, float* out, void* workspace,
                                  size_t workspace_bytes, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    BRN_CHECK_ARG(theta && grad && bandwidth && (out || rows == 0), "brn_svgd_direction: NULL pointer");
    BRN_CHECK_ARG(n >= 2 && d > 0, "brn_svgd_direction: need n >= 2 particles and d > 0 (got n=%d d=%d)", n, d);
    BRN_CHECK_ARG(row0 >= 0 && rows >= 0 && row0 + rows <= n, "brn_svgd_direction: bad row range [%d, %d) of %d", row0,
                  row0 + rows, n);
    SvgdWorkspace ws(workspace, n, d);
    BRN_CHECK_ARG(workspace && workspace_bytes >= ws.bytes, "workspace too small: %zu < %zu", workspace_bytes, ws.bytes);
    // tensor-core variant (tcgen05) for ensembles large enough to fill the tiles; BRN_SVGD_VARIANT=simt|tcgen05 forces one
    bool use_tc = n >= 512 && n % 4 == 0 && d + 1 <= SVGD_TC_BN && d >= 8;
    if (const char* env = getenv("BRN_SVGD_VARIANT")) {
        if (!strcmp(env, "simt")) use_tc = false;
        else if (!strcmp(env, "tcgen05")) {
            BRN_CHECK_ARG(d + 1 <= SVGD_TC_BN && n % 4 == 0, "BRN_SVGD_VARIANT=tcgen05 needs d < %d and n %% 4 == 0 (got d=%d n=%d)",
                          SVGD_TC_BN, d, n);
            use_tc = true;
        }
    }
    set_variant(use_tc ? "tcgen05" : "simt");
    const int sms = device_sm_count();
    {
        StageTimer st("svgd.pairwise_d2", stream);
        if (use_tc) {
            svgd_prep_theta_kernel<<<(n + 3) / 4, 128, 0, stream>>>(theta, n, d, ws.ldd, ws.th_hi, ws.th_lo, ws.sq);
            BRN_LAUNCH_OK("svgd_prep_theta_kernel");
            EpiD2::Params ep{ws.sq, ws.D2, n, n, 0};
            if (int e = launch_umma_nt<208, 16, EpiD2>(ws.th_hi, ws.th_lo, n, ws.ldd, ws.th_hi, ws.th_lo, n, ws.ldd, d, 0, 2, ep, stream))
                return e;
        } else {
            dim3 grid((n + SV_T - 1) / SV_T, (n + SV_T - 1) / SV_T);
            svgd_d2_kernel<<<grid, 256, 0, stream>>>(theta, n, d, ws.D2);
            BRN_LAUNCH_OK("svgd_d2_kernel");
        }
    }
    if (update_bandwidth) {
        StageTimer st("svgd.median_bandwidth", stream);
        const unsigned long long m = (unsigned long long)n * (unsigned long long)(n - 1) / 2ull;
        const unsigned long long k1 = (m - 1ull) / 2ull, k2 = m / 2ull;
        BRN_CUDA_OK(cudaMemsetAsync(ws.hist, 0, sizeof(unsigned int) * 4096, stream));
        const int64_t total = (int64_t)n * n;
        int64_t hblocks = (total + 255) / 256;
        if (hblocks > (int64_t)sms * 8) hblocks = (int64_t)sms * 8;
        const int hgrid = (int)hblocks;
        const int shifts[3] = {20, 8, 0}, nbits[3] = {12, 12, 8};
        for (int lv = 0; lv < 3; ++lv) {
            svgd_select_hist_kernel<<<hgrid, 256, sizeof(unsigned int) << nbits[lv], stream>>>(ws.D2, n, 0, n, shifts[lv], nbits[lv],
                                                                                             lv == 0, ws.st, ws.hist);
            BRN_LAUNCH_OK("svgd_select_hist_kernel");
            svgd_select_scan_kernel<<<1, SCAN_THREADS, 0, stream>>>(shifts[lv], nbits[lv], lv == 0, k1, ws.st, ws.hist);
            BRN_LAUNCH_OK("svgd_select_scan_kernel");
        }
        svgd_select_succ_kernel<<<hgrid, 256, 0, stream>>>(ws.D2, n, 0, n, ws.st);
        BRN_LAUNCH_OK("svgd_select_succ_kernel");
        svgd_bandwidth_kernel<<<1, 32, 0, stream>>>(ws.st, k2, n, bandwidth);
        BRN_LAUNCH_OK("svgd_bandwidth_kernel");
    }
    if (rows > 0 && use_tc) {
        StageTimer st("svgd.update", stream);
        dim3 grid((n + 31) / 32, (d + 1 + 31) / 32);
        svgd_prep_v_kernel<<<grid, 256, 0, stream>>>(theta, grad, n, d, bandwidth, ws.vt_hi, ws.vt_lo, ws.ldn);
        BRN_LAUNCH_OK("svgd_prep_v_kernel");
        BRN_CUDA_OK(cudaMemsetAsync(out, 0, sizeof(float) * (size_t)rows * d, stream));
        EpiSvgdOut::Params ep{out, theta, bandwidth, rows, d, row0};
        // A = D2 rows [rows][n] (plain fp32: exponentiated + split by the converter warps), B = V^T [d + 1][n]; K = n is split
        // over the grid (few output tiles) and the slices accumulate with atomics into the zeroed output
        if (int e = launch_umma_nt<SVGD_TC_BN, 16, EpiSvgdOut, 4, 1, 4>(ws.D2 + (size_t)row0 * n, nullptr, rows, n, ws.vt_hi, ws.vt_lo,
                                                                        d + 1, ws.ldn, n, 0, 2, ep, stream, true))
            return e;
    } else if (rows > 0) {
        StageTimer st("svgd.update", stream);
        const int row_tiles = (rows + SU_TI - 1) / SU_TI, d_chunks = (d + SU_TD - 1) / SU_TD;
        // ~8 CTAs (32 warps) per SM: with 2 the kernel ran at 7 warps per SM and 9.5 TFLOP/s (profiles/r1n_launches_svgd_summary.txt)
        int splits = (8 * sms) / (row_tiles * d_chunks);
        const int max_splits = (n + 4 * SU_TJ - 1) / (4 * SU_TJ);
        if (splits > max_splits) splits = max_splits;
        if (splits < 1) splits = 1;
        int j_per_split = ((n + splits - 1) / splits + SU_TJ - 1) / SU_TJ * SU_TJ;
        splits = (n + j_per_split - 1) / j_per_split;
        if (splits > 1) BRN_CUDA_OK(cudaMemsetAsync(out, 0, sizeof(float) * (size_t)rows * d, stream));
        dim3 grid(row_tiles, d_chunks, splits);
        svgd_update_kernel<<<grid, 128, 0, stream>>>(theta, grad, ws.D2, n, d, row0, rows, bandwidth, out, j_per_split);
        BRN_LAUNCH_OK("svgd_update_kernel");
    }
    return 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// K4b sharded over ranks (particles = rows): a rank keeps only ITS rows of D2 ([rows][n]), histograms its rows' part of the
// upper triangle, and the ranks add their histograms between the select passes -- the one real exchange step of the path.
// The collectives are the caller's (torch.distributed / NCCL on the buffers named by brn_svgd_sharded_offsets); this entry
// runs the device work between them:
//   phase 0: D2 rows, level-0 histogram                          -> all-reduce(SUM) hist
//   phase 1: scan level 0, level-1 histogram                     -> all-reduce(SUM) hist
//   phase 2: scan level 1, level-2 histogram                     -> all-reduce(SUM) hist
//   phase 3: scan level 2, successor pass (partial cnt_le, next) -> all-reduce(SUM) cnt_le, all-reduce(MIN) next
//   phase 4: bandwidth, update of the local rows
// Every rank ends with the bandwidth of the replicated evaluation bit for bit (integer histograms, identical scans).
extern "C" size_t brn_svgd_sharded_workspace_bytes(int n, int d, int rows) {
    if (n <= 0 || d <= 0 || rows < 0 || rows > n) return 0;
    return SvgdWorkspace(nullptr, n, d, rows).bytes;
}

extern "C" int brn_svgd_sharded_offsets(int n, int d, int rows, size_t* hist_off, size_t* hist_bytes, size_t* cnt_le_off,
                                        size_t* next_off) {
    BRN_CHECK_ARG(n > 0 && d > 0 && rows >= 0 && rows <= n && hist_off && hist_bytes && cnt_le_off && next_off,
                  "brn_svgd_sharded_offsets: bad arguments");
    SvgdWorkspace ws(nullptr, n, d, rows);
    *hist_off = ws.hist_off;
    *hist_bytes = sizeof(unsigned int) * 4096;
    *cnt_le_off = ws.st_off + offsetof(SelectState, cnt_le);
    *next_off = ws.st_off + offsetof(SelectState, next);
    return 0;
}

extern "C" int brn_svgd_sharded_phase(const float* theta, const float* grad, int n, int d, int row0, int rows, int phase,
                                      float* bandwidth, float* out, void* workspace, size_t workspace_bytes, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    BRN_CHECK_ARG(theta && grad && bandwidth && (out || rows == 0), "brn_svgd_sharded_phase: NULL pointer");
    BRN_CHECK_ARG(n >= 2 && d > 0, "brn_svgd_sharded_phase: need n >= 2 particles and d > 0 (got n=%d d=%d)", n, d);
    BRN_CHECK_ARG(row0 >= 0 && rows >= 0 && row0 + rows <= n, "brn_svgd_sharded_phase: bad row range [%d, %d) of %d", row0, row0 + rows, n);
    BRN_CHECK_ARG(phase >= 0 && phase <= 4, "brn_svgd_sharded_phase: phase %d (0..4)", phase);
    BRN_CHECK_ARG(n % 4 == 0 && d + 1 <= SVGD_TC_BN && d >= 8,
                  "brn_svgd_sharded_phase: the sharded evaluation runs on the tensor-core kernels (n %% 4 == 0, 8 <= d < %d; got n=%d d=%d)",
                  SVGD_TC_BN, n, d);
    SvgdWorkspace ws(workspace, n, d, rows);
    BRN_CHECK_ARG(workspace && workspace_bytes >= ws.bytes, "workspace too small: %zu < %zu", workspace_bytes, ws.bytes);
    set_variant("tcgen05");
    const int sms = device_sm_count();
    const unsigned long long m = (unsigned long long)n * (unsigned long long)(n - 1) / 2ull;
    const unsigned long long k1 = (m - 1ull) / 2ull, k2 = m / 2ull;
    int64_t hblocks = ((int64_t)rows * n + 255) / 256;
    if (hblocks > (int64_t)sms * 8) hblocks = (int64_t)sms * 8;
    if (hblocks < 1) hblocks = 1;
    const int hgrid = (int)hblocks;
    const int shifts[3] = {20, 8, 0}, nbits[3] = {12, 12, 8};
    if (phase == 0) {
        StageTimer st("svgd.pairwise_d2", stream);
        svgd_prep_theta_kernel<<<(n + 3) / 4, 128, 0, stream>>>(theta, n, d, ws.ldd, ws.th_hi, ws.th_lo, ws.sq);
        BRN_LAUNCH_OK("svgd_prep_theta_kernel");
        if (rows > 0) {
            EpiD2::Params ep{ws.sq, ws.D2, rows, n, row0};
            if (int e = launch_umma_nt<208, 16, EpiD2>(ws.th_hi + (size_t)row0 * ws.ldd, ws.th_lo + (size_t)row0 * ws.ldd, rows, ws.ldd,
                                                      ws.th_hi, ws.th_lo, n, ws.ldd, d, 0, 2, ep, stream))
                return e;
        }
        BRN_CUDA_OK(cudaMemsetAsync(ws.hist, 0, sizeof(unsigned int) * 4096, stream));
    }
    if (phase <= 3) {
        StageTimer st("svgd.median_bandwidth", stream);
        if (phase >= 1) {
            const int lv = phase - 1;
            svgd_select_scan_kernel<<<1, SCAN_THREADS, 0, stream>>>(shifts[lv], nbits[lv], lv == 0, k1, ws.st, ws.hist);
            BRN_LAUNCH_OK("svgd_select_scan_kernel");
        }
        if (phase <= 2) {
            if (rows > 0) {
                svgd_select_hist_kernel<<<hgrid, 256, sizeof(unsigned int) << nbits[phase], stream>>>(ws.D2, n, row0, rows, shifts[phase],
                                                                                                   nbits[phase], phase == 0, ws.st, ws.hist);
                BRN_LAUNCH_OK("svgd_select_hist_kernel");
            }
        } else if (rows > 0) {
            svgd_select_succ_kernel<<<hgrid, 256, 0, stream>>>(ws.D2, n, row0, rows, ws.st);
            BRN_LAUNCH_OK("svgd_select_succ_kernel");
        }
        return 0;
    }
    {
        StageTimer st("svgd.median_bandwidth", stream);
        svgd_bandwidth_kernel<<<1, 32, 0, stream>>>(ws.st, k2, n, bandwidth);
        BRN_LAUNCH_OK("svgd_bandwidth_kernel");
    }
    if (rows > 0) {
        StageTimer st("svgd.update", stream);
        dim3 grid((n + 31) / 32, (d + 1 + 31) / 32);
        svgd_prep_v_kernel<<<grid, 256, 0, stream>>>(theta, grad, n, d, bandwidth, ws.vt_hi, ws.vt_lo, ws.ldn);
        BRN_LAUNCH_OK("svgd_prep_v_kernel");
        BRN_CUDA_OK(cudaMemsetAsync(out, 0, sizeof(float) * (size_t)rows * d, stream));
        EpiSvgdOut::Params ep{out, theta, bandwidth, rows, d, row0};
        if (int e = launch_umma_nt<SVGD_TC_BN, 16, EpiSvgdOut, 4, 1, 4>(ws.D2, nullptr, rows, n, ws.vt_hi, ws.vt_lo, d + 1, ws.ldn, n, 0, 2,
                                                                        ep, stream, true))
            return e;
    }
    return 0;
}
