// One-shot all-reduce over NVLink / NVSwitch peer memory for the small variational-parameter gradient (SURVEY 8e: 636 KB at
// C3, 257 floats at C2 -- latency-bound, not bandwidth-bound).  Every rank copies its partial gradient into a symmetric
// buffer, raises a flag in every peer's flag array, waits for its own flags and then sums the peers' buffers straight out
// of their memory (loads over NVLink), in rank order -- so every rank obtains bit-identical sums.  One barrier per
// reduction: the buffers are double-buffered by the parity of an epoch counter that lives on the device, so the sequence
// can be captured in a CUDA graph and replayed (a rank can only pass the barrier of epoch e + 1 after every peer finished
// reading epoch e, hence nobody overwrites a buffer that is still being read).
// The reference has no collective at all (single process); this replaces what `ncclAllReduce` would do in SURVEY's proposal.
#include "common.cuh"
#include <algorithm>

namespace brn {

__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

// ONE kernel: (1) every block copies its slice of src into this rank's symmetric buffer of the coming epoch's parity and
// arrives on a local counter; (2) block 0 waits for all local blocks, then raises this rank's flag in every peer's flag
// array; (3) every block waits for all peers' flags of this epoch and sums the peers' buffers in rank order (the loads of
// one element from all peers are issued together: one NVLink round trip, not `world` of them).  status counts wait
// time-outs (a dead peer must not hang the GPU).  All blocks are co-resident (grid <= number of SMs).
// loss != NULL: the fp64 partial loss rides in the buffer's last quad as a (hi, lo) fp32 pair (elements n-4, n-3; the
// caller's src keeps that quad spare) and comes back summed -- no separate collective, no packing kernels.
constexpr int AR_MAX_WORLD = 16;

__global__ void __launch_bounds__(256)
allreduce_oneshot_kernel(const float* __restrict__ src, float* __restrict__ out, float* const* __restrict__ bufs,
                         unsigned long long* const* __restrict__ flags, int rank, int world, int64_t n,
                         unsigned long long* __restrict__ epoch, unsigned int* __restrict__ arrive, unsigned int* __restrict__ ticket,
                         unsigned int* __restrict__ status, double* __restrict__ loss) {
    const unsigned long long e = *epoch + 1ull;
    const int par = (int)(e & 1ull);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t tid0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    __shared__ int timed_out;
    if (threadIdx.x == 0) timed_out = 0;
    // (1) stage
    {
        float* dst = bufs[par * world + rank];
        for (int64_t i = tid0; i < n; i += stride) {
            float v = src[i];
            if (loss && i >= n - 4) {
                const double l = *loss;
                const float hi = (float)l;
                v = i == n - 4 ? hi : (i == n - 3 ? (float)(l - (double)hi) : 0.f);
            }
            dst[i] = v;
        }
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) atomicAdd(arrive, 1u);
    // (2) block 0: all local slices staged -> tell every peer
    if (blockIdx.x == 0) {
        if (threadIdx.x == 0) {
            const unsigned int want = (unsigned int)(e * gridDim.x);           // monotone across launches (same grid every call)
            long long spins = 0;
            while (*reinterpret_cast<volatile unsigned int*>(arrive) != want && ++spins < (1ll << 26)) {}
            __threadfence_system();
        }
        __syncthreads();
        if ((int)threadIdx.x < world) st_release_sys(flags[threadIdx.x] + rank, e);
    }
    // (3) wait for every peer's flag of this epoch
    if ((int)threadIdx.x < world) {
        const unsigned long long* f = flags[rank] + threadIdx.x;
        long long spins = 0;
        while (ld_acquire_sys(f) < e) {
            if (++spins > (1ll << 24)) { timed_out = 1; break; }   // ~ seconds: give up instead of hanging the device
            __nanosleep(32);
        }
    }
    __syncthreads();
    if (timed_out && threadIdx.x == 0) atomicAdd(status, 1u);
    const int64_t n4 = n / 4;
    for (int64_t q = tid0; q < n4; q += stride) {
        float4 v[AR_MAX_WORLD];
#pragma unroll
        for (int j = 0; j < AR_MAX_WORLD; ++j)
            if (j < world) v[j] = __ldcv(reinterpret_cast<const float4*>(bufs[par * world + j]) + q);     // never a stale L1 line
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int j = 0; j < AR_MAX_WORLD; ++j)
            if (j < world) { acc.x += v[j].x; acc.y += v[j].y; acc.z += v[j].z; acc.w += v[j].w; }
        reinterpret_cast<float4*>(out)[q] = acc;
        if (loss && q == n4 - 1) *loss = (double)acc.x + (double)acc.y;       // n % 4 == 0 when a loss rides along
    }
    for (int64_t i = n4 * 4 + tid0; i < n; i += stride) {
        float acc = 0.f;
        for (int j = 0; j < world; ++j) acc += __ldcv(bufs[par * world + j] + i);
        out[i] = acc;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(ticket, 1u) == gridDim.x - 1) {              // last block: publish the epoch for the next launch
            *ticket = 0u;
            *epoch = e;
        }
    }
}

}  // namespace brn

using namespace brn;

extern "C" int brn_allreduce_oneshot(const float* src, float* out, int64_t n, float* const* bufs_dev,
                                     unsigned long long* const* flags_dev, int rank, int world, uint64_t* state_dev,
                                     double* loss_inout, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    BRN_CHECK_ARG(src && out && bufs_dev && flags_dev && state_dev, "brn_allreduce_oneshot: NULL pointer");
    BRN_CHECK_ARG(n > 0 && world >= 1 && world <= 64 && rank >= 0 && rank < world, "brn_allreduce_oneshot: bad arguments n=%lld rank=%d world=%d",
                  (long long)n, rank, world);
    BRN_CHECK_ARG(((uintptr_t)out & 15) == 0, "brn_allreduce_oneshot: out must be 16-byte aligned");
    BRN_CHECK_ARG(!loss_inout || (n % 4 == 0 && n >= 4), "brn_allreduce_oneshot: a loss needs n %% 4 == 0 (its (hi, lo) pair uses the last quad)");
    BRN_CHECK_ARG(world <= AR_MAX_WORLD, "brn_allreduce_oneshot: at most %d ranks (got %d)", AR_MAX_WORLD, world);
    unsigned long long* epoch = reinterpret_cast<unsigned long long*>(state_dev);
    unsigned int* ticket = reinterpret_cast<unsigned int*>(state_dev + 1);
    unsigned int* status = ticket + 1;
    unsigned int* arrive = reinterpret_cast<unsigned int*>(state_dev + 2);
    // the grid is a pure function of n (the arrival counter assumes the same grid on every call of a given state)
    const int sms = device_sm_count();
    const unsigned grid = (unsigned)std::min<int64_t>((n / 4 + 255) / 256 + 1, sms);
    allreduce_oneshot_kernel<<<grid, 256, 0, stream>>>(src, out, bufs_dev, flags_dev, rank, world, n, epoch, arrive, ticket, status,
                                                       loss_inout);
    BRN_LAUNCH_OK("allreduce_oneshot_kernel");
    return 0;
}
