// K1: generic scalar-DAG ELBO -- fused reparameterised sampling, log-probabilities, two-axis reduction and the
// matching backward in ONE launch.  See include/brancher_cuda.h (brn_dag_elbo_fwd_bwd).
//
// The host (brancher_b200/lowering.py: DagPlan) flattens a (joint, posterior) pair whose variables are scalars
// (README AR(1), examples/logNormal_normal.py, examples/multivariate_regression.py ...) into a straight-line SSA
// program of `brn_dag_op`.  One thread evaluates the whole program for one (MC sample s, data row b) pair:
//   forward   values v[slot] in thread-local memory (every thread executes the same op sequence: no divergence)
//   reverse   adjoints in a second local array, walking the program backwards (reverse-mode AD by hand)
//   reduce    d loss / d param: shared-memory atomics per CTA, then one global atomic per parameter per CTA;
//             loss: warp-shuffle + shared reduction in fp64, one atomic per CTA.
// ACC_SAMPLE terms (latent log-probs, entropies) are counted once per sample (row 0 only), ACC_ROW terms (observed
// nodes: summed over the data axis, variables.py:513-514) for every row; loss = -(1/S_total) sum.
#include "common.cuh"

namespace brn {

enum DagOp : int32_t {
    DAG_CONST = BRN_DAG_CONST, DAG_PARAM = BRN_DAG_PARAM, DAG_DATA = BRN_DAG_DATA, DAG_EPS = BRN_DAG_EPS,
    DAG_ADD = BRN_DAG_ADD, DAG_SUB = BRN_DAG_SUB, DAG_MUL = BRN_DAG_MUL, DAG_DIV = BRN_DAG_DIV, DAG_NEG = BRN_DAG_NEG,
    DAG_POWI = BRN_DAG_POWI, DAG_EXP = BRN_DAG_EXP, DAG_LOG = BRN_DAG_LOG, DAG_LOG1P = BRN_DAG_LOG1P,
    DAG_SIGMOID = BRN_DAG_SIGMOID, DAG_SOFTPLUS = BRN_DAG_SOFTPLUS, DAG_TANH = BRN_DAG_TANH, DAG_SIN = BRN_DAG_SIN,
    DAG_COS = BRN_DAG_COS, DAG_RELU = BRN_DAG_RELU, DAG_SQRT = BRN_DAG_SQRT, DAG_ABS = BRN_DAG_ABS,
    DAG_CLAMP_UNIT = BRN_DAG_CLAMP_UNIT, DAG_NORMAL_LP = BRN_DAG_NORMAL_LP, DAG_NORMAL_ENTROPY = BRN_DAG_NORMAL_ENTROPY,
    DAG_ACC_SAMPLE = BRN_DAG_ACC_SAMPLE, DAG_ACC_ROW = BRN_DAG_ACC_ROW,
    DAG_UNIFORM_HEADER = BRN_DAG_UNIFORM_HEADER, DAG_LEVEL = BRN_DAG_LEVEL      // layout markers, not operations
};

constexpr int DAG_MAX_PARAMS = BRN_DAG_MAX_PARAMS;     // shared-memory gradient accumulators

__device__ __forceinline__ float dag_powi(float x, float p) { return powf(x, p); }

// One interpreted op costs a chain of dependent latencies (fetch -> decode -> operand loads -> ALU -> store), and a C1-sized
// problem has only ~10 warps to hide them, so the interpreter is built to shorten that chain:
//   * the program is packed to 16 bytes per op and staged in SHARED memory once per CTA (one broadcast LDS.128 per op);
//   * the next op is fetched while the current one executes, and both slot operands (and, in the reverse sweep, the
//     adjoint of dst) are loaded BEFORE the opcode switch so they overlap the indirect branch.
struct __align__(16) PackedOp { uint32_t w0, w1, c; float imm; };      // w0 = opcode | dst << 8 ; w1 = a | b << 16

//   * SMEM_FRAME (one warp per CTA, small programs): the value and adjoint frames live in SHARED memory, [slot][lane].
//     Thread-local frames are written once and read later (SSA), and local stores do not allocate in L1: every operand read
//     was an L2 round trip -- ~600 cycles per interpreted op at C1, where 10 warps cannot hide it (profiles/r1f_bench_ar1.json).
template <int MAXS, bool SMEM_FRAME>      // MAXS: value / adjoint slots per thread when the frames are thread-local
__global__ void __launch_bounds__(128)
dag_elbo_kernel(const brn_dag_op* __restrict__ ops, int n_ops, int n_slots, const float* __restrict__ params, int n_params,
                const float* __restrict__ data, int n_cols, int B, const float* __restrict__ eps, int n_eps,
                brn_sample_range r, float* __restrict__ dparams, double* __restrict__ loss) {
    extern __shared__ __align__(16) unsigned char dag_smem[];
    PackedOp* sops = reinterpret_cast<PackedOp*>(dag_smem);                    // [n_ops]
    float* sgrad = reinterpret_cast<float*>(dag_smem + sizeof(PackedOp) * (size_t)n_ops);   // [n_params]
    __shared__ double red[32];
    float vloc[SMEM_FRAME ? 1 : MAXS];
    float aloc[SMEM_FRAME ? 1 : MAXS];
    // shared frames start after sgrad, 128-byte aligned; [slot][lane] -> conflict-free, one wavefront per access
    float* const fbase = reinterpret_cast<float*>(
        (reinterpret_cast<uintptr_t>(sgrad + n_params) + 127) & ~(uintptr_t)127) + threadIdx.x;
    float* const vsm = fbase;
    float* const asm_ = fbase + (size_t)n_slots * 32;
    auto V = [&](int i) -> float& {
        if constexpr (SMEM_FRAME) return vsm[i * 32];
        else return vloc[i];
    };
    auto A = [&](int i) -> float& {
        if constexpr (SMEM_FRAME) return asm_[i * 32];
        else return aloc[i];
    };
    const int last_slot = n_slots - 1;
    for (int i = threadIdx.x; i < n_params; i += blockDim.x) sgrad[i] = 0.f;
#pragma unroll 4
    for (int i = threadIdx.x; i < n_ops; i += blockDim.x) {
        const brn_dag_op o = ops[i];
        PackedOp q;
        q.w0 = (uint32_t)o.opcode | ((uint32_t)o.dst << 8);
        q.w1 = ((uint32_t)o.a & 0xffffu) | ((uint32_t)o.b << 16);
        q.c = (uint32_t)o.c;
        q.imm = o.imm;
        sops[i] = q;
    }
    __syncthreads();

    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t total = (int64_t)r.s_local * B;
    const bool active = gid < total;
    const int s = active ? (int)(gid / B) : 0, b = active ? (int)(gid - (int64_t)s * B) : 0;
    const float inv_S = 1.0f / (float)r.s_total;
    const int lane = threadIdx.x & 31;
    float acc = 0.f;

    struct Op { int opcode, flags, dst, a, b, c; float imm; };      // flags: fused accumulation of the result (1 sample, 2 row)
    auto decode = [](const uint4& w) {
        Op o;
        o.opcode = (int)(w.x & 0x3fu); o.flags = (int)((w.x >> 6) & 3u); o.dst = (int)(w.x >> 8);
        o.a = (int)(w.y & 0xffffu); o.b = (int)(w.y >> 16);
        o.c = (int)w.z; o.imm = __uint_as_float(w.w);
        return o;
    };
    auto fetch = [&](int i) { return *reinterpret_cast<const uint4*>(&sops[i]); };

    // value of one op (va, vb = the a / b slot operands, already loaded)
    auto fwd_op = [&](const Op& o, float va, float vb) -> float {
        float x = 0.f;
        switch (o.opcode) {
            case DAG_CONST: x = o.imm; break;
            case DAG_PARAM: x = params[o.a]; break;
            case DAG_DATA: x = data[(int64_t)b * n_cols + o.a]; break;
            case DAG_EPS:
                x = eps ? eps[(int64_t)s * n_eps + o.a] : philox_normal1(r.seed, philox_offset(r), (uint32_t)o.a, (uint32_t)(r.s0 + s), 0);
                break;
            case DAG_ADD: x = va + vb; break;
            case DAG_SUB: x = va - vb; break;
            case DAG_MUL: x = va * vb; break;
            case DAG_DIV: x = va / vb; break;
            case DAG_NEG: x = -va; break;
            case DAG_POWI: x = dag_powi(va, o.imm); break;
            case DAG_EXP: x = expf(va); break;
            case DAG_LOG: x = logf(va); break;
            case DAG_LOG1P: x = log1pf(va); break;
            case DAG_SIGMOID: x = sigmoidf(va); break;
            case DAG_SOFTPLUS: x = softplusf(va); break;
            case DAG_TANH: x = tanhf(va); break;
            case DAG_SIN: x = sinf(va); break;
            case DAG_COS: x = cosf(va); break;
            case DAG_RELU: x = fmaxf(va, 0.f); break;
            case DAG_SQRT: x = sqrtf(va); break;
            case DAG_ABS: x = fabsf(va); break;
            case DAG_CLAMP_UNIT: x = fminf(fmaxf(va, 1.17549435e-38f), 1.0f - 1.1920929e-07f); break;
            case DAG_NORMAL_LP: {      // torch Normal.log_prob: -((x-mu)^2)/(2 sigma^2) - log sigma - log sqrt(2 pi)
                const float df = va - vb, sg = V(o.c);
                x = -(df * df) / (2.f * (sg * sg)) - logf(sg) - BRN_HALF_LOG_2PI;
                break;
            }
            case DAG_NORMAL_ENTROPY: x = 0.5f + BRN_HALF_LOG_2PI + logf(va); break;
            case DAG_ACC_SAMPLE: if (b == 0) acc += va; break;
            case DAG_ACC_ROW: acc += va; break;
            default: break;
        }
        return x;
    };
    // adjoint propagation of one op: g = d loss / d dst; adds into this thread's adjoint copies of the operand slots
    auto bwd_op = [&](const Op& o, float g, float va, float vb) {
        switch (o.opcode) {
            case DAG_ACC_SAMPLE: if (b == 0) A(o.a) -= inv_S; break;
            case DAG_ACC_ROW: A(o.a) -= inv_S; break;
            case DAG_PARAM: if (g != 0.f) atomicAdd(&sgrad[o.a], g); break;
            case DAG_ADD: A(o.a) += g; A(o.b) += g; break;
            case DAG_SUB: A(o.a) += g; A(o.b) -= g; break;
            case DAG_MUL: A(o.a) += g * vb; A(o.b) += g * va; break;
            case DAG_DIV: {
                const float inv = 1.f / vb;
                A(o.a) += g * inv;
                A(o.b) -= g * V(o.dst) * inv;
                break;
            }
            case DAG_NEG: A(o.a) -= g; break;
            case DAG_POWI: A(o.a) += g * o.imm * dag_powi(va, o.imm - 1.f); break;
            case DAG_EXP: A(o.a) += g * V(o.dst); break;
            case DAG_LOG: A(o.a) += g / va; break;
            case DAG_LOG1P: A(o.a) += g / (1.f + va); break;
            case DAG_SIGMOID: { const float y = V(o.dst); A(o.a) += g * y * (1.f - y); break; }
            case DAG_SOFTPLUS: A(o.a) += g * (va > 20.f ? 1.f : sigmoidf(va)); break;
            case DAG_TANH: { const float y = V(o.dst); A(o.a) += g * (1.f - y * y); break; }
            case DAG_SIN: A(o.a) += g * cosf(va); break;
            case DAG_COS: A(o.a) -= g * sinf(va); break;
            case DAG_RELU: A(o.a) += va > 0.f ? g : 0.f; break;
            case DAG_SQRT: A(o.a) += g * 0.5f / V(o.dst); break;
            case DAG_ABS: A(o.a) += va >= 0.f ? g : -g; break;
            case DAG_CLAMP_UNIT: A(o.a) += (va >= 1.17549435e-38f && va <= 1.0f - 1.1920929e-07f) ? g : 0.f; break;
            case DAG_NORMAL_LP: {
                const float df = va - vb, sg = V(o.c), inv_var = 1.f / (sg * sg);
                const float t = g * df * inv_var;
                A(o.a) -= t;
                A(o.b) += t;
                A(o.c) += g * (df * df * inv_var - 1.f) / sg;
                break;
            }
            case DAG_NORMAL_ENTROPY: A(o.a) += g / va; break;
            default: break;     // CONST / DATA / EPS: leaves
        }
    };

    // ---- table layout: [UNIFORM_HEADER (a = entries that follow)] { [LEVEL (a = ops in this level, b = ops in the previous
    //      one)] ops... }*  then the per-sample ops.  Uniform ops depend on parameters and constants only.
    int u_begin = 0, u_end = 0;
    int n_eps_ops = 0, n_data_ops = 0;                  // leading EPS / DATA ops of the per-sample segment (header fields b, c)
    if ((sops[0].w0 & 0xffu) == DAG_UNIFORM_HEADER) {
        u_begin = 1; u_end = 1 + (int)(sops[0].w1 & 0xffffu);
        n_eps_ops = (int)(sops[0].w1 >> 16); n_data_ops = (int)sops[0].c;
    }
    const int s_begin = SMEM_FRAME ? u_end : 0;       // thread-local frames: every thread evaluates the uniform ops itself

    int last_marker = -1;
    if constexpr (SMEM_FRAME) {
        // ---------------- uniform forward: ONE evaluation per CTA, the lanes of the warp take the ops of a dependency level in
        // parallel (a serial walk costs one full op latency per op, and C1 has too few warps to hide any of it); each result
        // is broadcast into all 32 lane copies of its slot (rotated: conflict-free)
        for (int i = u_begin; i < u_end;) {
            const int cnt = (int)(sops[i].w1 & 0xffffu);
            for (int k = i + 1 + lane; k <= i + cnt; k += 32) {
                const Op o = decode(fetch(k));
                const float x = fwd_op(o, V(min(o.a, last_slot)), V(min(o.b, last_slot)));
                float* row = vsm - lane + (size_t)o.dst * 32;
#pragma unroll 8
                for (int j = 0; j < 32; ++j) row[(j + lane) & 31] = x;
            }
            __syncwarp();
            last_marker = i;
            i += cnt + 1;
        }
        for (int i = 0; i < n_slots; ++i) A(i) = 0.f;       // every lane (idle lanes help in the uniform reverse sweep)
    }

    if (active) {
        // ---------------- leaves first (shared-memory frames): the noise draws and the data loads of a thread are independent
        // of each other, so two branch-free loops let them overlap instead of paying one full latency per interpreted op
        int s_fwd = s_begin;
        if constexpr (SMEM_FRAME) {
#pragma unroll 4
            for (int i = s_fwd; i < s_fwd + n_eps_ops; ++i) {
                const Op o = decode(fetch(i));
                V(o.dst) = eps ? eps[(int64_t)s * n_eps + o.a] : philox_normal1(r.seed, philox_offset(r), (uint32_t)o.a, (uint32_t)(r.s0 + s), 0);
            }
            s_fwd += n_eps_ops;
#pragma unroll 4
            for (int i = s_fwd; i < s_fwd + n_data_ops; ++i) {
                const Op o = decode(fetch(i));
                V(o.dst) = data[(int64_t)b * n_cols + o.a];
            }
            s_fwd += n_data_ops;
        }
        // ---------------- forward
        uint4 nxt = fetch(min(s_fwd, n_ops - 1));
        for (int i = s_fwd; i < n_ops; ++i) {
            const Op o = decode(nxt);
            nxt = fetch(min(i + 1, n_ops - 1));
            if (o.opcode >= DAG_UNIFORM_HEADER) continue;       // layout markers (thread-local frames walk the whole table)
            const float va = V(min(o.a, last_slot)), vb = V(min(o.b, last_slot));       // operand loads overlap the branch
            const float x = fwd_op(o, va, vb);
            V(o.dst) = x;
            if (o.flags) {                                      // ACC_SAMPLE / ACC_ROW of this result, fused by the host
                if ((o.flags & 1) && b == 0) acc += x;
                if (o.flags & 2) acc += x;
            }
        }
        // ---------------- reverse: d loss / d slot, loss = -(1/S) * acc
        if constexpr (!SMEM_FRAME)
            for (int i = 0; i < n_slots; ++i) A(i) = 0.f;
        nxt = fetch(n_ops - 1);
        for (int i = n_ops - 1; i >= s_fwd; --i) {          // (leaves have no operands: nothing to propagate)
            const Op o = decode(nxt);
            nxt = fetch(max(i - 1, 0));
            if (o.opcode >= DAG_UNIFORM_HEADER) continue;
            float g = A(o.dst);
            if (o.flags) {
                if ((o.flags & 1) && b == 0) g -= inv_S;
                if (o.flags & 2) g -= inv_S;
            }
            const float va = V(min(o.a, last_slot)), vb = V(min(o.b, last_slot));
            bwd_op(o, g, va, vb);
        }
    }

    if constexpr (SMEM_FRAME) {
        // ---------------- uniform reverse, levels in descending order: the adjoint of a uniform slot is the SUM of its 32 lane
        // copies (per-sample consumers and later uniform ops both add into per-lane copies)
        __syncwarp();
        for (int i = last_marker; i >= u_begin;) {
            const int cnt = (int)(sops[i].w1 & 0xffffu), prev = (int)(sops[i].w1 >> 16);
            for (int k = i + 1 + lane; k <= i + cnt; k += 32) {
                const Op o = decode(fetch(k));
                const float* row = asm_ - lane + (size_t)o.dst * 32;
                float g = 0.f;
#pragma unroll 8
                for (int j = 0; j < 32; ++j) g += row[(j + lane) & 31];
                bwd_op(o, g, V(min(o.a, last_slot)), V(min(o.b, last_slot)));
            }
            __syncwarp();
            if (i == u_begin) break;
            i -= prev + 1;
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n_params; i += blockDim.x) {
        const float gsum = sgrad[i];
        if (gsum != 0.f) atomicAdd(&dparams[i], gsum);
    }
    double tot = block_sum<double>((double)acc, red);
    if (threadIdx.x == 0) atomicAdd(loss, -tot * (double)inv_S);
}

}  // namespace brn

using namespace brn;

extern "C" int brn_dag_elbo_fwd_bwd(const brn_dag_op* ops, int n_ops, int n_slots, const float* params, int n_params,
                                    const float* data, int n_cols, int n_rows, const float* eps, int n_eps,
                                    const brn_sample_range* r, float* dparams, double* loss, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    BRN_CHECK_ARG(ops && r && loss, "brn_dag_elbo_fwd_bwd: NULL pointer");
    BRN_CHECK_ARG(n_ops > 0 && n_slots > 0 && n_slots <= BRN_DAG_MAX_SLOTS, "brn_dag_elbo_fwd_bwd: n_slots=%d outside (0, %d]",
                  n_slots, BRN_DAG_MAX_SLOTS);
    BRN_CHECK_ARG(n_params >= 0 && n_params <= DAG_MAX_PARAMS, "brn_dag_elbo_fwd_bwd: n_params=%d exceeds %d", n_params, DAG_MAX_PARAMS);
    BRN_CHECK_ARG(n_params == 0 || (params && dparams), "brn_dag_elbo_fwd_bwd: NULL parameter pointer");
    BRN_CHECK_ARG(n_rows >= 1 && n_cols >= 0 && (n_cols == 0 || data), "brn_dag_elbo_fwd_bwd: bad data block rows=%d cols=%d", n_rows,
                  n_cols);
    if (int e = check_sample_range(*r)) return e;
    if (r->s_local == 0) return 0;
    set_variant("simt");
    StageTimer st("dag.fused", stream);
    const int64_t total = (int64_t)r->s_local * n_rows;
    // The value/adjoint arrays live in thread-local memory (2 * n_slots lines of 128 B per warp).  Small problems (the
    // README AR(1): 300 samples) run ONE WARP PER CTA so that (a) the work spreads over as many SMs as there are warps and
    // (b) each SM's L1 holds its warp's whole local frame -- with 128-thread CTAs the frame of ~700 slots spilled to L2 and
    // every interpreted op paid an L2 round trip (563 us per evaluation, measured; profiles/r1e_bench_ar1.json).
    const int block = total <= (int64_t)32 * 148 * 8 ? 32 : 128;
    const unsigned grid = (unsigned)((total + block - 1) / block);
    size_t smem = sizeof(PackedOp) * (size_t)n_ops + sizeof(float) * (size_t)(n_params > 0 ? n_params : 1);
    BRN_CHECK_ARG(smem <= 96 * 1024, "brn_dag_elbo_fwd_bwd: program of %d ops does not fit in shared memory", n_ops);
    BRN_CHECK_ARG(n_cols <= 65536 && n_eps <= 65536, "brn_dag_elbo_fwd_bwd: n_cols=%d / n_eps=%d exceed the 16-bit operand field",
                  n_cols, n_eps);
    // frames in shared memory when one warp per CTA is used and both frames fit beside the program
    const size_t frames = 2 * (size_t)n_slots * 32 * sizeof(float) + 128;
    const bool smem_frame = block == 32 && smem + frames <= 220 * 1024;
    if (smem_frame) smem += frames;
#define BRN_DAG_LAUNCH(MAXS, SF)                                                                                          \
    {                                                                                                                     \
        BRN_CUDA_OK(cudaFuncSetAttribute(dag_elbo_kernel<MAXS, SF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        dag_elbo_kernel<MAXS, SF><<<grid, block, smem, stream>>>(ops, n_ops, n_slots, params, n_params, data, n_cols, n_rows, \
                                                                 eps, n_eps, *r, dparams, loss);                           \
    }
    if (smem_frame) BRN_DAG_LAUNCH(128, true)
    else if (n_slots <= 128) BRN_DAG_LAUNCH(128, false)
    else if (n_slots <= 512) BRN_DAG_LAUNCH(512, false)
    else BRN_DAG_LAUNCH(BRN_DAG_MAX_SLOTS, false)
#undef BRN_DAG_LAUNCH
    BRN_LAUNCH_OK("dag_elbo_kernel");
    return 0;
}
