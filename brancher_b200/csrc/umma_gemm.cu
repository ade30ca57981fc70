// Host side of the tcgen05 GEMM building block: TMA descriptor encoding (driver entry point resolved at
// run time -- no link-time libcuda dependency), the TF32 hi/lo splitter, and a plain GEMM entry point
// (brn_gemm_nt_3xtf32) used by the tests to validate the tensor-core path in isolation.
#include "umma_gemm.cuh"
#include <stdio.h>

#include <cudaTypedefs.h>
#include <stdlib.h>

namespace brn {

static PFN_cuTensorMapEncodeTiled_v12000 get_encode_fn() {
    static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
    }
    return fn;
}

int make_tmap_2d_f32(CUtensorMap* out, const float* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows,
                     uint32_t box_cols, bool atom32) {
    auto fn = get_encode_fn();
    if (!fn) { set_error("cuTensorMapEncodeTiled is not available from the driver"); return -4; }
    if (((uintptr_t)base & 15) || (ld * sizeof(float)) % 16) {
        set_error("TMA operand must be 16-byte aligned with a 16-byte multiple row pitch (base=%p ld=%llu)", (const void*)base,
                  (unsigned long long)ld);
        return -1;
    }
    cuuint64_t gdim[2] = {cols, rows};
    cuuint64_t gstr[1] = {ld * sizeof(float)};
    if (box_cols != 32 && box_cols != 16) { set_error("TMA box must be 32 or 16 floats wide (got %u)", box_cols); return -1; }
    cuuint32_t box[2] = {box_cols, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), gdim, gstr, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE,
                    // atom32: 128-byte swizzle at 32-byte granularity, the layout tf32 operands need to be read MN-major
                    atom32 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : (box_cols == 32 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B),
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows=%llu cols=%llu ld=%llu box=%u)",
                                       (int)r, (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)ld, box_rows);
        return -4; }
    return 0;
}

int make_tmap_2d_f16(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows,
                     uint32_t box_cols) {
    auto fn = get_encode_fn();
    if (!fn) { set_error("cuTensorMapEncodeTiled is not available from the driver"); return -4; }
    if (((uintptr_t)base & 15) || (ld * 2) % 16) {
        set_error("TMA operand must be 16-byte aligned with a 16-byte multiple row pitch (base=%p ld=%llu halves)", base,
                  (unsigned long long)ld);
        return -1;
    }
    cuuint64_t gdim[2] = {cols, rows};
    cuuint64_t gstr[1] = {ld * 2};
    if (box_cols != 64 && box_cols != 32) { set_error("fp16 TMA box must be 64 or 32 elements wide (got %u)", box_cols); return -1; }
    cuuint32_t box[2] = {box_cols, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), gdim, gstr, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, box_cols == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled (fp16) failed with CUresult %d (rows=%llu cols=%llu ld=%llu box=%u)",
                                       (int)r, (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)ld, box_rows);
        return -4; }
    return 0;
}

// hi/lo split of src [rows][cols] (row pitch lds) into dst_hi/dst_lo [rows][ldd]; optionally also the
// transposed pair [cols][ldt].  Pad columns (>= cols) are not touched (TMA never reads them: the tensor map's
// extent is `cols`).
__global__ void split_tf32_kernel(const float* __restrict__ src, int64_t lds, int rows, int cols, float* __restrict__ hi,
                                  float* __restrict__ lo, int64_t ldd, float* __restrict__ thi, float* __restrict__ tlo,
                                  int64_t ldt) {
    __shared__ float th[32][33], tl[32][33];
    const int c0 = blockIdx.y * 32, r0 = blockIdx.x * 32;       // row tiles on grid.x: rows may be millions
    const int tx = threadIdx.x, ty = threadIdx.y;       // 32 x 8
    for (int i = ty; i < 32; i += 8) {
        int r = r0 + i, c = c0 + tx;
        float h = 0.f, l = 0.f;
        if (r < rows && c < cols) {
            umma::split_tf32(src[(int64_t)r * lds + c], h, l);
            if (hi) {               // row-major pair optional (an operand read in place needs only the transposed pair)
                hi[(int64_t)r * ldd + c] = h;
                lo[(int64_t)r * ldd + c] = l;
            }
        }
        th[i][tx] = h; tl[i][tx] = l;
    }
    if (thi == nullptr) return;
    __syncthreads();
    for (int i = ty; i < 32; i += 8) {
        int c = c0 + i, r = r0 + tx;
        if (r < rows && c < cols) {
            thi[(int64_t)c * ldt + r] = th[tx][i];
            tlo[(int64_t)c * ldt + r] = tl[tx][i];
        }
    }
}

// plain transpose: dst [cols][ldt] = src [rows][lds]^T  (operands the GEMM splits on the fly, SPLIT mask in umma_gemm.cuh)
__global__ void transpose_f32_kernel(const float* __restrict__ src, int64_t lds, int rows, int cols, float* __restrict__ dst,
                                     int64_t ldt) {
    __shared__ float t[32][33];
    const int c0 = blockIdx.y * 32, r0 = blockIdx.x * 32;
    const int tx = threadIdx.x, ty = threadIdx.y;       // 32 x 8
    for (int i = ty; i < 32; i += 8) {
        const int r = r0 + i, c = c0 + tx;
        t[i][tx] = (r < rows && c < cols) ? src[(int64_t)r * lds + c] : 0.f;
    }
    __syncthreads();
    for (int i = ty; i < 32; i += 8) {
        const int c = c0 + i, r = r0 + tx;
        if (r < rows && c < cols) dst[(int64_t)c * ldt + r] = t[tx][i];
    }
}

int launch_transpose_f32(const float* src, int64_t lds, int rows, int cols, float* dst, int64_t ldt, cudaStream_t stream) {
    if (rows <= 0 || cols <= 0) return 0;
    dim3 grid((rows + 31) / 32, (cols + 31) / 32), block(32, 8);
    transpose_f32_kernel<<<grid, block, 0, stream>>>(src, lds, rows, cols, dst, ldt);
    BRN_LAUNCH_OK("transpose_f32_kernel");
    return 0;
}

int launch_split_tf32(const float* src, int64_t lds, int rows, int cols, float* hi, float* lo, int64_t ldd, float* thi,
                      float* tlo, int64_t ldt, cudaStream_t stream) {
    if (rows <= 0 || cols <= 0) return 0;
    dim3 grid((rows + 31) / 32, (cols + 31) / 32), block(32, 8);
    split_tf32_kernel<<<grid, block, 0, stream>>>(src, lds, rows, cols, hi, lo, ldd, thi, tlo, ldt);
    BRN_LAUNCH_OK("split_tf32_kernel");
    return 0;
}

}  // namespace brn

using namespace brn;

static size_t pad4(size_t n) { return (n + 3) / 4 * 4; }

extern "C" size_t brn_gemm_nt_workspace_bytes(int M, int N, int K) {
    size_t ld = pad4((size_t)K);
    return sizeof(float) * 2 * ((size_t)M * ld + (size_t)N * ld) + 4096;
}

// D[M][N] (row-major, ldd = N) = A[M][K] . B[N][K]^T with 3xTF32 on tcgen05.
extern "C" int brn_gemm_nt_3xtf32(const float* A, const float* B, float* D, int M, int N, int K, void* workspace,
                                  size_t workspace_bytes, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    BRN_CHECK_ARG(A && B && D && workspace, "brn_gemm_nt_3xtf32: NULL pointer");
    BRN_CHECK_ARG(M > 0 && N > 0 && K > 0, "brn_gemm_nt_3xtf32: bad shape");
    BRN_CHECK_ARG(workspace_bytes >= brn_gemm_nt_workspace_bytes(M, N, K), "brn_gemm_nt_3xtf32: workspace too small");
    const size_t ld = pad4((size_t)K);
    float* base = reinterpret_cast<float*>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    float *Ah = base, *Al = Ah + (size_t)M * ld, *Bh = Al + (size_t)M * ld, *Bl = Bh + (size_t)N * ld;
    if (int e = launch_split_tf32(A, K, M, K, Ah, Al, ld, nullptr, nullptr, 0, stream)) return e;
    if (int e = launch_split_tf32(B, K, N, K, Bh, Bl, ld, nullptr, nullptr, 0, stream)) return e;
    set_variant("tcgen05");
    constexpr int drain = 2;      // TMEM accumulation chain of 2 x 32 words of K between register drains (umma_gemm.cuh)
    // N tile / epilogue warps: 224 x 8 by default; BRN_GEMM_BN = 208 | 256 select the other instantiated shapes (tile-shape
    // measurements, profiles/gemm_bn_sweep.py)
    int bn = 224;
    if (const char* env = getenv("BRN_GEMM_BN")) bn = atoi(env);
    const int cpt = bn == 256 ? 64 : bn / 2;          // accumulator columns per epilogue thread = one output block
    EpiStore::Params ep;
    ep.out = D; ep.rows = M; ep.row_stride = N; ep.col_stride = 1; ep.blk_stride = cpt; ep.blk_valid = cpt;
    ep.col_limit = N; ep.total_blks = (N + cpt - 1) / cpt;
    StageTimer st("gemm.umma", stream);
    if (const char* env = getenv("BRN_UMMA_BK"))
        if (atoi(env) == 32) return launch_umma_nt<224, 32, EpiStore>(Ah, Al, M, ld, Bh, Bl, N, ld, K, 0, drain, ep, stream);
    if (bn == -208 || bn == -209) {
        // MMA-rate measurements (profiles/gemm_bn_sweep.py): null epilogue; -209 issues the same byte streams as kind::f16
        // (the fp32 words read as pairs of halves: numerically meaningless, but twice the MACs per instruction)
        EpiNull::Params en{D};
        if (bn == -208) return launch_umma_nt<208, 16, EpiNull>(Ah, Al, M, ld, Bh, Bl, N, ld, K, 0, drain, en, stream);
        return launch_umma_nt_kind<208, 16, EpiNull, 8, 0, 4, 1>(Ah, Al, M, 2 * ld, Bh, Bl, N, 2 * ld, 2 * K, 0, drain, en, stream);
    }
    if (bn == -300) {
        // MN-major operands (launch_umma_tn_plain): D = At^T . Bt for the transposed plain copies At [K][M], Bt [K][N]
        const size_t ldm = pad4((size_t)M), ldn = pad4((size_t)N);
        float *At = base, *Bt = At + (size_t)K * ldm;
        BRN_CHECK_ARG((size_t)K * (ldm + ldn) * sizeof(float) + 4096 <= workspace_bytes, "workspace too small for the MN-major test");
        if (int e = launch_transpose_f32(A, K, M, K, At, ldm, stream)) return e;
        if (int e = launch_transpose_f32(B, K, N, K, Bt, ldn, stream)) return e;
        constexpr int cptm = 64;
        ep.blk_stride = cptm; ep.blk_valid = cptm; ep.total_blks = (N + cptm - 1) / cptm;
        return launch_umma_tn_plain<128, 16, EpiStore, 8, 4>(At, M, ldm, Bt, N, ldn, K, 0, drain, ep, stream);
    }
    if (bn == 208) return launch_umma_nt<208, 16, EpiStore>(Ah, Al, M, ld, Bh, Bl, N, ld, K, 0, drain, ep, stream);
    if (bn == 256) return launch_umma_nt<256, 16, EpiStore, 16>(Ah, Al, M, ld, Bh, Bl, N, ld, K, 0, drain, ep, stream);
    return launch_umma_nt<224, 16, EpiStore>(Ah, Al, M, ld, Bh, Bl, N, ld, K, 0, drain, ep, stream);
}
