// K1a: mean-field Normal sampling, prior log-prob, analytic entropy and their pathwise gradients.
// HBM-bound elementwise + sample-axis reduction; one thread owns 4 consecutive elements (one Philox
// call) and walks the local samples, so every global access is coalesced across the warp.
#include "meanfield.cuh"

namespace brn {

__global__ void philox_fill_kernel(float* __restrict__ out, int64_t ld, int64_t numel, uint32_t var_id,
                                   brn_sample_range r) {
    int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int s = blockIdx.y;
    if (q * 4 >= numel) return;
    Normal4 n = philox_normal4(r.seed, philox_offset(r), var_id, (uint32_t)(r.s0 + s), (uint32_t)q);
    float* o = out + (int64_t)s * ld + q * 4;
#pragma unroll
    for (int j = 0; j < 4; ++j)
        if (q * 4 + j < numel) o[j] = n.v[j];
}

int launch_philox_fill(float* out, int64_t ld, int64_t numel, uint32_t var_id, const brn_sample_range& r,
                       cudaStream_t stream) {
    if (numel <= 0 || r.s_local <= 0) return 0;
    int64_t quads = (numel + 3) / 4;
    dim3 grid((unsigned)((quads + 255) / 256), (unsigned)r.s_local);
    philox_fill_kernel<<<grid, 256, 0, stream>>>(out, ld, numel, var_id, r);
    BRN_LAUNCH_OK("philox_fill_kernel");
    return 0;
}

__global__ void sample_weights_kernel(const float* __restrict__ mu, const float* __restrict__ rho,
                                      const float* __restrict__ eps, int64_t lde, float* __restrict__ W, int64_t ldw,
                                      int64_t numel) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int s = blockIdx.y;
    if (i >= numel) return;
    float sg = softplusf(rho[i]);
    W[(int64_t)s * ldw + i] = __fmaf_rn(sg, eps[(int64_t)s * lde + i], mu[i]);
}

int launch_sample_weights(const float* mu, const float* rho, const float* eps, int64_t lde, float* W, int64_t ldw,
                          int64_t numel, int s_local, cudaStream_t stream) {
    if (numel <= 0 || s_local <= 0) return 0;
    dim3 grid((unsigned)((numel + 255) / 256), (unsigned)s_local);
    sample_weights_kernel<<<grid, 256, 0, stream>>>(mu, rho, eps, lde, W, ldw, numel);
    BRN_LAUNCH_OK("sample_weights_kernel");
    return 0;
}

// One thread per quad of elements; loops over the local samples.
__global__ void __launch_bounds__(256)
mf_finalize_kernel(brn_mf_var v, const float* __restrict__ eps, int64_t lde, const float* __restrict__ gw,
                   const float* __restrict__ gwe, brn_sample_range r, int with_prior, double* __restrict__ loss) {
    __shared__ double red[32];
    int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double elbo_thread = 0.0;
    if (q * 4 < v.numel) {
        const int nvalid = (int)min((int64_t)4, v.numel - q * 4);
        float mu[4], sg[4], a[4], inv_b2[4], lp[4], dmu_acc[4], dsg_acc[4], rho[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            int64_t i = q * 4 + j;
            bool ok = j < nvalid;
            mu[j] = ok ? v.mu[i] : 0.f;
            rho[j] = ok ? v.rho[i] : 0.f;
            sg[j] = softplusf(rho[j]);
            a[j] = (ok && !v.tied) ? v.prior_loc[i] : 0.f;
            float b = (ok && !v.tied) ? v.prior_scale[i] : 1.f;
            inv_b2[j] = 1.0f / (b * b);
            lp[j] = 0.f; dmu_acc[j] = 0.f; dsg_acc[j] = 0.f;
        }
        if (with_prior) {
            for (int s = 0; s < r.s_local; ++s) {
                float e[4];
                if (eps) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) e[j] = j < nvalid ? eps[(int64_t)s * lde + q * 4 + j] : 0.f;
                } else {
                    Normal4 n = philox_normal4(r.seed, philox_offset(r), v.var_id, (uint32_t)(r.s0 + s), (uint32_t)q);
#pragma unroll
                    for (int j = 0; j < 4; ++j) e[j] = n.v[j];
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (v.tied) {
                        // log N(w; mu, sigma) with w = mu + sigma*eps  ==  -eps^2/2 - log sigma - c ;
                        // d/dmu and the eps-dependent part of d/dsigma cancel identically.
                        lp[j] += -0.5f * e[j] * e[j];
                    } else {
                        float d = __fmaf_rn(sg[j], e[j], mu[j]) - a[j];
                        float gwp = -d * inv_b2[j];            // d logp / d w
                        lp[j] += 0.5f * d * gwp;               // -d^2 / (2 b^2)
                        dmu_acc[j] += gwp;
                        dsg_acc[j] += gwp * e[j];
                    }
                }
            }
        }
        const float inv_S = 1.0f / (float)r.s_total;
        const float frac = (float)r.s_local * inv_S;   // share of the per-sample constants owned by this rank
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (j >= nvalid) continue;
            int64_t i = q * 4 + j;
            float dE_dmu = 0.f, dE_dsg = 0.f;
            if (with_prior) {
                float log_sg = logf(sg[j]);
                float entropy = 0.5f + BRN_HALF_LOG_2PI + log_sg;
                float lp_const = v.tied ? (-log_sg - BRN_HALF_LOG_2PI)
                                        : (-logf(v.prior_scale[i]) - BRN_HALF_LOG_2PI);
                elbo_thread += (double)(lp[j] * inv_S) + (double)(frac * (lp_const + entropy));
                dE_dmu = dmu_acc[j] * inv_S;
                // tied: prior -1/sigma and entropy +1/sigma cancel
                dE_dsg = v.tied ? 0.f : (dsg_acc[j] * inv_S + frac / sg[j]);
            }
            if (gw) dE_dmu += gw[i] * inv_S;
            if (gwe) dE_dsg += gwe[i] * inv_S;
            v.dmu[i] += -dE_dmu;
            v.drho[i] += -dE_dsg * sigmoidf(rho[j]);
        }
    }
    double tot = block_sum<double>(elbo_thread, red);
    if (threadIdx.x == 0 && with_prior) atomicAdd(loss, -tot);
}

int launch_mf_finalize(const brn_mf_var& var, const float* eps, int64_t lde, const float* gw, const float* gwe,
                       const brn_sample_range& r, int with_prior, double* loss, cudaStream_t stream) {
    if (var.numel <= 0) return 0;
    if (!eps && var.eps) { eps = var.eps; lde = var.numel; }
    int64_t quads = (var.numel + 3) / 4;
    unsigned grid = (unsigned)((quads + 255) / 256);
    mf_finalize_kernel<<<grid, 256, 0, stream>>>(var, eps, lde, gw, gwe, r, with_prior, loss);
    BRN_LAUNCH_OK("mf_finalize_kernel");
    return 0;
}

__global__ void __launch_bounds__(256)
reduce_over_samples_kernel(const float* __restrict__ dW, int64_t ld, const float* __restrict__ eps, int64_t lde,
                           float* __restrict__ gw, float* __restrict__ gwe, int64_t numel, int s_local) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= numel) return;
    float a0 = 0.f, a1 = 0.f, b0 = 0.f, b1 = 0.f;
    int s = 0;
    for (; s + 1 < s_local; s += 2) {
        float d0 = dW[(int64_t)s * ld + i], d1 = dW[(int64_t)(s + 1) * ld + i];
        float e0 = eps[(int64_t)s * lde + i], e1 = eps[(int64_t)(s + 1) * lde + i];
        a0 += d0; a1 += d1;
        b0 = __fmaf_rn(d0, e0, b0); b1 = __fmaf_rn(d1, e1, b1);
    }
    if (s < s_local) {
        float d0 = dW[(int64_t)s * ld + i], e0 = eps[(int64_t)s * lde + i];
        a0 += d0; b0 = __fmaf_rn(d0, e0, b0);
    }
    gw[i] = a0 + a1;
    gwe[i] = b0 + b1;
}

int launch_reduce_over_samples(const float* dW, int64_t ld, const float* eps, int64_t lde, float* gw, float* gwe,
                               int64_t numel, int s_local, cudaStream_t stream) {
    if (numel <= 0) return 0;
    unsigned grid = (unsigned)((numel + 255) / 256);
    reduce_over_samples_kernel<<<grid, 256, 0, stream>>>(dW, ld, eps, lde, gw, gwe, numel, s_local);
    BRN_LAUNCH_OK("reduce_over_samples_kernel");
    return 0;
}

// ---------------------------------------------------------------------------------------------
// stage 5, parallel version
// ---------------------------------------------------------------------------------------------
// CTA = 32 quads (128 consecutive elements: every load of a warp is one 512-byte row segment) x 8 sample groups; sample group y
// walks samples y, y+8, ...; the 8 partial sums per element are combined in shared memory and STORED -- each element is owned
// by exactly one CTA, so there are neither atomics nor a zeroing pass.  (The first version split the sample axis over
// the grid and issued 16 global atomics per thread: 5.1 M atomics per C3 evaluation, 53 us for 160 MB.)
struct MfMulti {
    brn_mf_var v[4];
    int64_t off[4];
    int n;
};

constexpr int MF_QUADS = 32, MF_SGROUPS = 8;

// FUSE: the owning CTA also finalises its 128 elements (several variables back to back, MfMulti) instead of storing the
// statistics for a second kernel: one launch and one dependent-launch gap less per evaluation.
template <bool FUSE>
__global__ void __launch_bounds__(MF_QUADS * MF_SGROUPS)
mf_stats_kernel(const float* __restrict__ eps, int64_t lde, const float* __restrict__ dW, int64_t ldd, int64_t numel,
                int64_t npad, brn_sample_range r, uint32_t var_id, int vec, int64_t philox_quads,
                float* __restrict__ stats, MfMulti m, int with_prior, double* __restrict__ loss) {
    __shared__ float4 part[4][MF_SGROUPS][MF_QUADS];
    __shared__ double red[32];
    const int tx = threadIdx.x & (MF_QUADS - 1), ty = threadIdx.x / MF_QUADS;
    const int64_t q = (int64_t)blockIdx.x * MF_QUADS + tx;
    const bool live = q * 4 < numel;
    const int nvalid = live ? (int)min((int64_t)4, numel - q * 4) : 0;
    vec = vec && nvalid == 4;          // `vec` = pitches/bases allow float4; the ragged last quad goes scalar
    float gw[4] = {0.f, 0.f, 0.f, 0.f}, gwe[4] = {0.f, 0.f, 0.f, 0.f}, e1[4] = {0.f, 0.f, 0.f, 0.f}, e2[4] = {0.f, 0.f, 0.f, 0.f};
    if (live && vec && eps && dW && q >= philox_quads) {
        // common case (stored noise, vectorisable): explicit batches of 8 samples = 16 independent 16-byte loads in flight per
        // thread before the first use
        const float4* e4p = reinterpret_cast<const float4*>(eps + q * 4);
        const float4* d4p = reinterpret_cast<const float4*>(dW + q * 4);
        const int64_t le4 = lde / 4, ld4 = ldd / 4;
        for (int s0 = ty; s0 < r.s_local; s0 += 8 * MF_SGROUPS) {
            float4 e4[8], d4[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int s = s0 + u * MF_SGROUPS;
                if (s < r.s_local) {
                    e4[u] = __ldg(e4p + (int64_t)s * le4);
                    d4[u] = __ldg(d4p + (int64_t)s * ld4);
                } else {
                    e4[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                    d4[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const float e[4] = {e4[u].x, e4[u].y, e4[u].z, e4[u].w}, d[4] = {d4[u].x, d4[u].y, d4[u].z, d4[u].w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    gw[j] += d[j];
                    gwe[j] = __fmaf_rn(d[j], e[j], gwe[j]);
                    e1[j] += e[j];
                    e2[j] = __fmaf_rn(e[j], e[j], e2[j]);
                }
            }
        }
    } else if (live) {
#pragma unroll 8
        for (int s = ty; s < r.s_local; s += MF_SGROUPS) {
            float e[4], d[4] = {0.f, 0.f, 0.f, 0.f};
            if (eps && q >= philox_quads) {     // quads below philox_quads are regenerated (never stored): same counters as the sampler
                if (vec) {
                    float4 t = *reinterpret_cast<const float4*>(eps + (int64_t)s * lde + q * 4);
                    e[0] = t.x; e[1] = t.y; e[2] = t.z; e[3] = t.w;
                } else {
#pragma unroll
                    for (int j = 0; j < 4; ++j) e[j] = j < nvalid ? eps[(int64_t)s * lde + q * 4 + j] : 0.f;
                }
            } else {
                Normal4 n = philox_normal4(r.seed, philox_offset(r), var_id, (uint32_t)(r.s0 + s), (uint32_t)q);
#pragma unroll
                for (int j = 0; j < 4; ++j) e[j] = j < nvalid ? n.v[j] : 0.f;
            }
            if (dW) {
                if (vec) {
                    float4 t = *reinterpret_cast<const float4*>(dW + (int64_t)s * ldd + q * 4);
                    d[0] = t.x; d[1] = t.y; d[2] = t.z; d[3] = t.w;
                } else {
#pragma unroll
                    for (int j = 0; j < 4; ++j) d[j] = j < nvalid ? dW[(int64_t)s * ldd + q * 4 + j] : 0.f;
                }
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                gw[j] += d[j];
                gwe[j] = __fmaf_rn(d[j], e[j], gwe[j]);
                e1[j] += e[j];
                e2[j] = __fmaf_rn(e[j], e[j], e2[j]);
            }
        }
    }
    part[0][ty][tx] = make_float4(gw[0], gw[1], gw[2], gw[3]);
    part[1][ty][tx] = make_float4(gwe[0], gwe[1], gwe[2], gwe[3]);
    part[2][ty][tx] = make_float4(e1[0], e1[1], e1[2], e1[3]);
    part[3][ty][tx] = make_float4(e2[0], e2[1], e2[2], e2[3]);
    __syncthreads();
    if constexpr (FUSE) {
        double elbo = 0.0;
        const int el = threadIdx.x;
        const int64_t g = (int64_t)blockIdx.x * MF_QUADS * 4 + el;
        if (el < MF_QUADS * 4 && g < numel) {
            float st4[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                float acc = 0.f;
#pragma unroll
                for (int y = 0; y < MF_SGROUPS; ++y) acc += reinterpret_cast<const float*>(&part[k][y][el >> 2])[el & 3];
                st4[k] = acc;
            }
            int k = 0;
#pragma unroll
            for (int j = 1; j < 4; ++j)
                if (j < m.n && g >= m.off[j]) k = j;
            const int64_t i = g - m.off[k];
            if (i < m.v[k].numel) elbo = mf_finalize_element(m.v[k], i, dW ? st4[0] : 0.f, dW ? st4[1] : 0.f, st4[2], st4[3], r, with_prior);
        }
        const double tot = block_sum<double>(elbo, red);
        if (threadIdx.x == 0 && with_prior) atomicAdd(loss, -tot);
        return;
    }
    // 4 statistics x 128 elements per CTA: thread t sums the 8 group partials of (statistic t / 128, element t % 128)
    for (int t = threadIdx.x; t < 4 * MF_QUADS * 4; t += MF_QUADS * MF_SGROUPS) {
        const int k = t / (MF_QUADS * 4), el = t % (MF_QUADS * 4);
        const int64_t i = (int64_t)blockIdx.x * MF_QUADS * 4 + el;
        if (i >= numel || (k < 2 && !dW)) continue;
        float acc = 0.f;
#pragma unroll
        for (int y = 0; y < MF_SGROUPS; ++y) acc += reinterpret_cast<const float*>(&part[k][y][el >> 2])[el & 3];
        stats[(int64_t)k * npad + i] = acc;
    }
}

__global__ void __launch_bounds__(256)
mf_finalize2_kernel(brn_mf_var v, const float* __restrict__ stats, int64_t npad, brn_sample_range r, int with_prior,
                    double* __restrict__ loss) {
    __shared__ double red[32];
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double elbo_thread = 0.0;
    if (i < v.numel) {
        const float mu = v.mu[i], rho = v.rho[i], sg = softplusf(rho);
        const float gw = stats[i], gwe = stats[npad + i], e1 = stats[2 * npad + i], e2 = stats[3 * npad + i];
        const float inv_S = 1.0f / (float)r.s_total, n = (float)r.s_local, frac = n * inv_S;
        float dE_dmu = gw * inv_S, dE_dsg = gwe * inv_S;
        if (with_prior) {
            const float log_sg = logf(sg);
            const float entropy = 0.5f + BRN_HALF_LOG_2PI + log_sg;
            if (v.tied) {
                // log N(w; mu, sigma), w = mu + sigma*eps  ==  -eps^2/2 - log sigma - c ; its mu- and sigma-gradients
                // cancel against themselves / the entropy identically.
                elbo_thread = (double)(-0.5f * e2 * inv_S) + (double)(frac * (entropy - log_sg - BRN_HALF_LOG_2PI));
            } else {
                const float a = v.prior_loc[i], b = v.prior_scale[i], inv_b2 = 1.0f / (b * b);
                const float c0 = mu - a;
                // sum_s (c0 + sg*eps_s)^2, sum_s (c0 + sg*eps_s), sum_s (c0 + sg*eps_s)*eps_s from (n, e1, e2)
                const float sd2 = n * c0 * c0 + 2.f * c0 * sg * e1 + sg * sg * e2;
                const float sd = n * c0 + sg * e1;
                const float sde = c0 * e1 + sg * e2;
                elbo_thread = (double)(-0.5f * sd2 * inv_b2 * inv_S) + (double)(frac * (entropy - logf(b) - BRN_HALF_LOG_2PI));
                dE_dmu += -sd * inv_b2 * inv_S;
                dE_dsg += -sde * inv_b2 * inv_S + frac / sg;
            }
        }
        v.dmu[i] += -dE_dmu;
        v.drho[i] += -dE_dsg * sigmoidf(rho);
    }
    double tot = block_sum<double>(elbo_thread, red);
    if (threadIdx.x == 0 && with_prior) atomicAdd(loss, -tot);
}

int launch_mf_reduce_finalize(const brn_mf_var& var, const float* eps, int64_t lde, const float* dW, int64_t ldd,
                              float* stats, const brn_sample_range& r, int with_prior, double* loss, cudaStream_t stream) {
    if (var.numel <= 0) return 0;
    if (!eps && var.eps) { eps = var.eps; lde = var.numel; }
    const int64_t npad = (var.numel + 3) / 4 * 4;
    // the stats kernel stores every statistic it owns; zero only what it will not write
    if (r.s_local <= 0 || !dW) BRN_CUDA_OK(cudaMemsetAsync(stats, 0, sizeof(float) * 4 * npad, stream));
    if (r.s_local > 0) {
        const int64_t quads = npad / 4;
        const int vec = (!eps || (((uintptr_t)eps % 16 == 0) && lde % 4 == 0)) &&
                        (!dW || (((uintptr_t)dW % 16 == 0) && ldd % 4 == 0));
        const unsigned grid = (unsigned)((quads + MF_QUADS - 1) / MF_QUADS);
        mf_stats_kernel<false><<<grid, MF_QUADS * MF_SGROUPS, 0, stream>>>(eps, lde, dW, ldd, var.numel, npad, r, var.var_id, vec, 0, stats,
                                                                           MfMulti(), 0, nullptr);
        BRN_LAUNCH_OK("mf_stats_kernel");
    }
    mf_finalize2_kernel<<<(unsigned)((var.numel + 255) / 256), 256, 0, stream>>>(var, stats, npad, r, with_prior, loss);
    BRN_LAUNCH_OK("mf_finalize2_kernel");
    return 0;
}

// ---------------------------------------------------------------------------------------------
// stage 5 for several variables laid out back to back in one [S][ld] block (the BNN workspace): ONE stats launch
// over the concatenated element range and ONE finalize launch that looks the variable up per element.
// ---------------------------------------------------------------------------------------------

__global__ void __launch_bounds__(256)
mf_finalize_multi_kernel(MfMulti m, const float* __restrict__ stats, int64_t npad, int64_t total, brn_sample_range r,
                         int with_prior, double* __restrict__ loss) {
    __shared__ double red[32];
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double elbo_thread = 0.0;
    if (g < total) {
        int k = 0;
#pragma unroll
        for (int j = 1; j < 4; ++j)
            if (j < m.n && g >= m.off[j]) k = j;
        const brn_mf_var& v = m.v[k];
        const int64_t i = g - m.off[k];
        if (i < v.numel) {
            const float mu = v.mu[i], rho = v.rho[i], sg = softplusf(rho);
            const float gw = stats[g], gwe = stats[npad + g], e1 = stats[2 * npad + g], e2 = stats[3 * npad + g];
            const float inv_S = 1.0f / (float)r.s_total, n = (float)r.s_local, frac = n * inv_S;
            float dE_dmu = gw * inv_S, dE_dsg = gwe * inv_S;
            if (with_prior) {
                const float log_sg = logf(sg);
                const float entropy = 0.5f + BRN_HALF_LOG_2PI + log_sg;
                if (v.tied) {
                    elbo_thread = (double)(-0.5f * e2 * inv_S) + (double)(frac * (entropy - log_sg - BRN_HALF_LOG_2PI));
                } else {
                    const float a = v.prior_loc[i], b = v.prior_scale[i], inv_b2 = 1.0f / (b * b);
                    const float c0 = mu - a;
                    const float sd2 = n * c0 * c0 + 2.f * c0 * sg * e1 + sg * sg * e2;
                    const float sd = n * c0 + sg * e1;
                    const float sde = c0 * e1 + sg * e2;
                    elbo_thread = (double)(-0.5f * sd2 * inv_b2 * inv_S) + (double)(frac * (entropy - logf(b) - BRN_HALF_LOG_2PI));
                    dE_dmu += -sd * inv_b2 * inv_S;
                    dE_dsg += -sde * inv_b2 * inv_S + frac / sg;
                }
            }
            v.dmu[i] += -dE_dmu;
            v.drho[i] += -dE_dsg * sigmoidf(rho);
        }
    }
    double tot = block_sum<double>(elbo_thread, red);
    if (threadIdx.x == 0 && with_prior) atomicAdd(loss, -tot);
}

int launch_mf_reduce_finalize_multi(const brn_mf_var* vars, const int64_t* offs, int nvars, int64_t total, const float* eps,
                                    int64_t lde, const float* dW, int64_t ldd, float* stats, const brn_sample_range& r,
                                    int with_prior, double* loss, cudaStream_t stream, int64_t philox_numel0) {
    // philox_numel0 > 0: the noise of the first philox_numel0 elements (variable 0, which must start at offset 0) was
    // never stored -- the stats kernel regenerates it from the same Philox counters the sampler used.
    if (philox_numel0 > 0 && (offs[0] != 0 || philox_numel0 % 4 != 0 || philox_numel0 > vars[0].numel)) {
        set_error("launch_mf_reduce_finalize_multi: bad regenerated-noise range %lld", (long long)philox_numel0);
        return -1;
    }
    if (nvars <= 0 || nvars > 4 || total <= 0) { set_error("launch_mf_reduce_finalize_multi: bad variable count %d", nvars); return -1; }
    const int64_t npad = (total + 3) / 4 * 4;
    MfMulti m;
    m.n = nvars;
    for (int k = 0; k < 4; ++k) {
        m.v[k] = vars[k < nvars ? k : nvars - 1];
        m.off[k] = offs[k < nvars ? k : nvars - 1];
    }
    if (r.s_local > 0) {
        // statistics + finalisation in ONE launch: every element is owned by exactly one CTA
        const int64_t quads = npad / 4;
        const int vec = (((uintptr_t)eps % 16 == 0) && lde % 4 == 0) && (!dW || (((uintptr_t)dW % 16 == 0) && ldd % 4 == 0));
        const unsigned grid = (unsigned)((quads + MF_QUADS - 1) / MF_QUADS);
        mf_stats_kernel<true><<<grid, MF_QUADS * MF_SGROUPS, 0, stream>>>(eps, lde, dW, ldd, total, npad, r, vars[0].var_id, vec,
                                                                          philox_numel0 / 4, stats, m, with_prior, loss);
        BRN_LAUNCH_OK("mf_stats_kernel");
        return 0;
    }
    BRN_CUDA_OK(cudaMemsetAsync(stats, 0, sizeof(float) * 4 * npad, stream));
    mf_finalize_multi_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(m, stats, npad, total, r, with_prior, loss);
    BRN_LAUNCH_OK("mf_finalize_multi_kernel");
    return 0;
}

// several small variables sampled in one launch: eps (injected or Philox) -> eps_out[s*ld + off_k + i] and
// W[s*ld + off_k + i] = mu + softplus(rho) * eps
struct SampleMulti {
    const float* mu[4]; const float* rho[4]; const float* eps_in[4];
    int64_t off[4], numel[4];
    uint32_t var_id[4];
    int n;
};

__global__ void __launch_bounds__(256)
sample_multi_kernel(SampleMulti m, int64_t total, float* __restrict__ eps_out, float* __restrict__ W, int64_t ld,
                    brn_sample_range r, float* __restrict__ grad_zero) {
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int s = blockIdx.y;
    if (g >= total) return;
    int k = 0;
    int64_t base = 0;
    bool found = false;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        if (!found && j < m.n) {
            if (g < base + m.numel[j]) { k = j; found = true; }
            else base += m.numel[j];
        }
    }
    if (!found) return;
    const int64_t i = g - base;
    const float e = m.eps_in[k] ? m.eps_in[k][(int64_t)s * m.numel[k] + i]
                                : philox_normal1(r.seed, philox_offset(r), m.var_id[k], (uint32_t)(r.s0 + s), i);
    const int64_t o = (int64_t)s * ld + m.off[k] + i;
    eps_out[o] = e;
    W[o] = __fmaf_rn(softplusf(m.rho[k][i]), e, m.mu[k][i]);
    if (grad_zero) grad_zero[o] = 0.f;        // per-sample gradient slot of the same element (accumulated into later): saves a memset node
}

int launch_sample_multi(const brn_mf_var* vars, const int64_t* offs, int nvars, float* eps_out, float* W, int64_t ld,
                        const brn_sample_range& r, cudaStream_t stream, float* grad_zero) {
    if (nvars <= 0 || nvars > 4) { set_error("launch_sample_multi: bad variable count %d", nvars); return -1; }
    SampleMulti m;
    m.n = nvars;
    int64_t total = 0;
    for (int k = 0; k < 4; ++k) {
        const int kk = k < nvars ? k : nvars - 1;
        m.mu[k] = vars[kk].mu; m.rho[k] = vars[kk].rho; m.eps_in[k] = vars[kk].eps;
        m.off[k] = offs[kk]; m.numel[k] = vars[kk].numel; m.var_id[k] = vars[kk].var_id;
        if (k < nvars) total += vars[k].numel;
    }
    if (total <= 0 || r.s_local <= 0) return 0;
    dim3 grid((unsigned)((total + 255) / 256), (unsigned)r.s_local);
    sample_multi_kernel<<<grid, 256, 0, stream>>>(m, total, eps_out, W, ld, r, grad_zero);
    BRN_LAUNCH_OK("sample_multi_kernel");
    return 0;
}

}  // namespace brn

using namespace brn;

static int check_range(const brn_sample_range* r) {
    BRN_CHECK_ARG(r != nullptr, "sample range is NULL");
    return check_sample_range(*r);
}

extern "C" int brn_philox_normal_fill(float* out, int64_t numel, uint32_t var_id, const brn_sample_range* r,
                                      void* stream) {
    if (check_range(r)) return -1;
    BRN_CHECK_ARG(out != nullptr && numel >= 0, "brn_philox_normal_fill: bad output");
    return launch_philox_fill(out, numel, numel, var_id, *r, (cudaStream_t)stream);
}

extern "C" int brn_mf_normal_prior_entropy(const brn_mf_var* var, const float* lik_gw, const float* lik_gwe,
                                           const brn_sample_range* r, double* loss, void* stream) {
    if (check_range(r)) return -1;
    BRN_CHECK_ARG(var && var->mu && var->rho && var->dmu && var->drho && loss, "brn_mf_normal_prior_entropy: NULL pointer");
    BRN_CHECK_ARG(var->tied || (var->prior_loc && var->prior_scale), "prior_loc/prior_scale required when not tied");
    return launch_mf_finalize(*var, nullptr, 0, lik_gw, lik_gwe, *r, 1, loss, (cudaStream_t)stream);
}
