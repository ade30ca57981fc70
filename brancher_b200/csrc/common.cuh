// Shared device helpers: error reporting, Philox4x32-10 + Box-Muller, stable elementwise math,
// warp/block reductions.  sm_100a only.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <string.h>

#include "../../include/brancher_cuda.h"

namespace brn {

// ---------------------------------------------------------------------------------------------
// host-side error plumbing
// ---------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
void set_variant(const char* name);
void count_launch(int n);

#define BRN_CHECK_ARG(cond, ...)                 \
    do {                                         \
        if (!(cond)) {                           \
            brn::set_error(__VA_ARGS__);         \
            return -1;                           \
        }                                        \
    } while (0)

#define BRN_CUDA_OK(expr)                                                                    \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess) {                                                             \
            brn::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return -2;                                                                       \
        }                                                                                    \
    } while (0)

#define BRN_LAUNCH_OK(name)                                                                  \
    do {                                                                                     \
        cudaError_t _e = cudaGetLastError();                                                 \
        if (_e != cudaSuccess) {                                                             \
            brn::set_error("launch of %s failed: %s", name, cudaGetErrorString(_e));         \
            return -3;                                                                       \
        }                                                                                    \
        brn::count_launch(1);                                                                \
    } while (0)

// SM count of the current device, read on every call (the caller may switch devices between calls)
inline int device_sm_count() {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return sms;
}

// Cuts a workspace into consecutive pieces, each rounded up to 256 bytes.  With base == NULL it only counts: `off` is then
// the number of bytes the same sequence of requests needs.
struct WorkspaceCarver {
    void* base; size_t off = 0;
    explicit WorkspaceCarver(void* b) : base(b) {}
    char* bytes(size_t n) {
        char* p = base ? static_cast<char*>(base) + off : nullptr;
        off += (n + 255) / 256 * 256;
        return p;
    }
    float* operator()(size_t nfloat) { return reinterpret_cast<float*>(bytes(nfloat * sizeof(float))); }
};

inline int check_sample_range(const brn_sample_range& r) {
    BRN_CHECK_ARG(r.s_local >= 0 && r.s_total > 0 && r.s0 >= 0 && r.s0 + r.s_local <= r.s_total,
                  "bad sample range s0=%d s_local=%d s_total=%d", r.s0, r.s_local, r.s_total);
    return 0;
}

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. 2011).  key = seed, counter = (i/4, global sample, var_id, offset).
// One call -> 4 x u32 -> 4 standard normals (two Box-Muller pairs), element i uses lane i%4.
// All arithmetic below is spelled with explicit rounding intrinsics so that every kernel that inlines
// it produces bit-identical normals (no context-dependent FMA contraction).
// ---------------------------------------------------------------------------------------------
struct Philox4 {
    uint32_t x, y, z, w;
};

__device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                 uint32_t k0, uint32_t k1) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(M0, c0), lo0 = M0 * c0;
        uint32_t hi1 = __umulhi(M1, c2), lo1 = M1 * c2;
        uint32_t n0 = hi1 ^ c1 ^ k0;
        uint32_t n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += W0; k1 += W1;
    }
    return Philox4{c0, c1, c2, c3};
}

// u32 -> uniform in (0,1): (x>>8 + 0.5) * 2^-24
__device__ __forceinline__ float u01(uint32_t x) {
    return __fmaf_rn((float)(x >> 8), 5.9604644775390625e-8f, 2.98023223876953125e-8f);
}

__device__ __forceinline__ void box_muller(uint32_t a, uint32_t b, float& z0, float& z1) {
    float u1 = u01(a), u2 = u01(b);
    float r = __fsqrt_rn(__fmul_rn(-2.0f, __logf(u1)));
    float s, c;
    __sincosf(__fmul_rn(6.283185307179586f, u2), &s, &c);
    z0 = __fmul_rn(r, c);
    z1 = __fmul_rn(r, s);
}

struct Normal4 {
    float v[4];
};

// four normals for elements 4*q .. 4*q+3 of variable `var_id`, global sample `s`
__device__ __forceinline__ Normal4 philox_normal4(uint64_t seed, uint64_t offset, uint32_t var_id, uint32_t s,
                                                  uint32_t q) {
    // offset's high word is folded into the key so that 2^64 iterations never collide
    Philox4 p = philox4x32_10(q, s, var_id, (uint32_t)offset, (uint32_t)seed,
                              (uint32_t)(seed >> 32) ^ (uint32_t)(offset >> 32));
    Normal4 n;
    box_muller(p.x, p.y, n.v[0], n.v[1]);
    box_muller(p.z, p.w, n.v[2], n.v[3]);
    return n;
}

// counter word 3: the by-value offset plus, when given, an offset the device owns (brn_sample_range.offset_dev) -- lets a
// CUDA-graph-captured iteration draw fresh noise on every replay without re-recording its kernel arguments
__device__ __forceinline__ uint64_t philox_offset(const brn_sample_range& r) {
    return r.offset + (r.offset_dev ? __ldg(reinterpret_cast<const unsigned long long*>(r.offset_dev)) : 0ull);
}

__device__ __forceinline__ float philox_normal1(uint64_t seed, uint64_t offset, uint32_t var_id, uint32_t s,
                                                int64_t i) {
    Normal4 n = philox_normal4(seed, offset, var_id, s, (uint32_t)(i >> 2));
    return n.v[i & 3];
}

// ---------------------------------------------------------------------------------------------
// stable scalar math (matches torch's formulas: softplus threshold 20, log-sigmoid via log1p)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float softplusf(float x) {      // torch.nn.functional.softplus(beta=1, threshold=20)
    return x > 20.0f ? x : log1pf(expf(x));
}
__device__ __forceinline__ float sigmoidf(float x) {
    return 1.0f / (1.0f + expf(-x));
}
// log(1 + exp(x)) without the torch threshold: max(x,0) + log1p(exp(-|x|))  (Binomial/Bernoulli normaliser)
__device__ __forceinline__ float log1pexpf(float x) {
    return fmaxf(x, 0.0f) + log1pf(expf(-fabsf(x)));
}

#define BRN_HALF_LOG_2PI 0.9189385332046727f

// ---------------------------------------------------------------------------------------------
// reductions
// ---------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// block-wide sum; result valid in thread 0.  `scratch` >= 32 elements of shared memory.
template <typename T>
__device__ __forceinline__ T block_sum(T v, T* scratch) {
    int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) scratch[wid] = v;
    __syncthreads();
    T r = (T)0;
    if (wid == 0) {
        r = lane < nw ? scratch[lane] : (T)0;
        r = warp_sum(r);
    }
    return r;
}

}  // namespace brn

// ---------------------------------------------------------------------------------------------
// optional per-stage timing (CUDA events on the launch stream) and launch counting, for bench.py
// ---------------------------------------------------------------------------------------------
namespace brn {
void count_launch(int n);
int wait_data_ready(cudaStream_t stream);    // consumes the event of brn_set_data_ready_event (no-op when none is pending)

struct StageTimer {      // RAII: records an event pair around a stage when profiling is enabled
    int slot;
    cudaStream_t stream;
    StageTimer(const char* name, cudaStream_t s);
    ~StageTimer();
};
}  // namespace brn
