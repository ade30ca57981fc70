/* brancher_cuda.h -- C ABI of the B200-native Monte-Carlo ELBO / pathwise-gradient hot path.
 *
 * The reference (LucaAmbrogioni/Brancher, pure Python) has NO FFI / plugin interface; its boundary for
 * this path is the Python object API (SURVEY.md §8b).  This header is the native boundary the Python
 * host mirror (`brancher_b200`, same class / method names as `brancher`) binds with ctypes.  Each entry
 * point states which reference code it replaces (paths relative to the reference repo).
 *
 * Conventions
 *  - every pointer is a DEVICE pointer owned by the caller (torch); fp32 unless stated; row-major.
 *  - `stream` is a cudaStream_t (0 = legacy default stream).  Calls only enqueue work.
 *  - return 0 on success, <0 on error; `brn_last_error()` gives the message (thread-local).
 *  - MC samples are indexed globally: this process evaluates samples [s0, s0+S_local) of S_total, so
 *    results are invariant to how samples are sharded over GPUs (SURVEY.md §8e).  Every output is a
 *    PARTIAL already scaled by 1/S_total and ACCUMULATED (+=) into caller-zeroed buffers; summing the
 *    partials of all ranks (NCCL all-reduce, done by the host) gives loss = -ELBO and d loss/d param.
 *  - noise: `eps` != NULL -> caller-injected standard normals, layout [S_local, numel] per variable;
 *    `eps` == NULL -> Philox4x32-10 keyed by (seed), counter (element/4, global sample, var_id, offset)
 *    + Box-Muller, bit-identical to what `brn_philox_normal_fill` writes.
 */
#ifndef BRANCHER_CUDA_H
#define BRANCHER_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BRN_ABI_VERSION 5

/* One mean-field Normal variational variable  q(w) = N(mu, softplus(rho))  together with the Normal
 * prior p(w) = N(prior_loc, prior_scale) of the same name.
 * Replaces: NormalVariable(loc, scale, name, learnable=True) (brancher/standard_variables.py:133-145),
 * its auto-created roots `<name>_loc`, `<name>_scale` with scale = softplus(rho)
 * (standard_variables.py:57-68, geometric_ranges.py:48-57), Normal rsample / log_prob / entropy
 * (distributions.py:111-124,170-181,155-168 -> torch.distributions.Normal).
 * tied != 0 reproduces the reference's root-NAME collision: p's hyper-parameter roots take q's values
 * (utilities.py:282-309, variables.py:367-371), so log p(w) = N(w; mu, sigma) and prior_* are ignored. */
typedef struct brn_mf_var {
    const float* mu;          /* [numel]            `<name>_loc`   parameter                       */
    const float* rho;         /* [numel]            `<name>_scale` parameter (sigma = softplus)    */
    const float* prior_loc;   /* [numel] or NULL when tied                                         */
    const float* prior_scale; /* [numel] or NULL when tied                                         */
    const float* eps;         /* [S_local, numel] injected noise, or NULL for Philox               */
    float*       dmu;         /* [numel]  += d loss / d mu   (partial, scaled)                     */
    float*       drho;        /* [numel]  += d loss / d rho  (partial, scaled)                     */
    int64_t      numel;
    uint32_t     var_id;      /* Philox stream id of this variable                                 */
    int32_t      tied;
} brn_mf_var;

/* Which MC samples this call evaluates and how noise is produced. */
typedef struct brn_sample_range {
    int32_t  s0;        /* first global sample index                      */
    int32_t  s_local;   /* samples evaluated by this call                 */
    int32_t  s_total;   /* global number of samples (the .mean() divisor, gradient_estimators.py:44) */
    int32_t  _pad;
    uint64_t seed;      /* Philox key                                     */
    uint64_t offset;    /* Philox counter word 3 (iteration number)       */
    const uint64_t* offset_dev; /* optional DEVICE scalar added to `offset` when the noise is drawn (NULL: none): a
                                 * CUDA-graph-captured iteration bumps it on the device instead of re-recording arguments */
} brn_sample_range;

int         brn_abi_version(void);
const char* brn_last_error(void);
/* name of the kernel variant the last compute call dispatched to ("simt", "tcgen05", ...) */
const char* brn_last_variant(void);

/* eps[s - s0, i] for s in [s0, s0+s_local), i in [0, numel): exactly the normals the fused kernels
 * generate for (seed, offset, var_id).  Replaces torch.distributions.normal._standard_normal as called by
 * Normal.rsample under distributions.py:122. */
int brn_philox_normal_fill(float* out, int64_t numel, uint32_t var_id, const brn_sample_range* r, void* stream);

/* K1a -- prior + entropy of mean-field Normal variables, forward and backward in one launch:
 *   loss  += -(1/S_total) sum_{s local} [ sum_i log N(w_si; prior) + sum_i H(N(mu_i, sigma_i)) ]
 *   dmu/drho += matching gradients (through w = mu + sigma*eps, through the entropy and -- when tied --
 *   through the prior's own parameters).
 * If lik_gw / lik_gwe are non-NULL they hold the likelihood stage's raw sums
 *   gw[i] = sum_s d ll_s / d w_si,  gwe[i] = sum_s eps_si * d ll_s / d w_si   (ELBO direction, unscaled)
 * and are folded in:  dmu -= gw/S_total,  drho -= sigmoid(rho) * gwe/S_total.
 * Replaces: RandomVariable.calculate_log_probability for the weight nodes (variables.py:486-520),
 * Variable._get_entropy (variables.py:156-162) and their autograd backward. */
int brn_mf_normal_prior_entropy(const brn_mf_var* var, const float* lik_gw, const float* lik_gwe,
                                const brn_sample_range* r, double* loss, void* stream);

/* K3 -- Bayesian neural network P-H-C (tanh), Categorical(logits) likelihood over B observed rows:
 *   per sample s: W1_s = mu+sigma*eps (H x P), b1_s (H), W2_s (C x H), b2_s (C)
 *   ll_s = sum_b log_softmax(W2_s tanh(W1_s x_b + b1_s) + b2_s)[y_b]
 *   loss += -(1/S_total) sum_s ll_s ; plus prior/entropy of the four variables (K1a folded in);
 *   dmu/drho of vars[0..3] = (weights1, b1, weights2, b2) accumulated.
 * Replaces the whole graph walk of estimate_log_model_evidence (variables.py:843-870) for the model of
 * development_playgrounds/MNIST_bayesian_neural_network.py:26-57: _get_sample (variables.py:527-570),
 * _apply_link's (S*B, H, P) materialisation + bmm (variables.py:436-449), CategoricalDistribution
 * log-prob (distributions.py:294-311), the data-axis sum (variables.py:513-514), the sample-axis mean
 * (gradient_estimators.py:44) and loss.backward() (inference.py:100).
 * X [B,P] fp32, y [B] int32 labels.  workspace: brn_bnn_workspace_bytes() bytes of scratch. */
size_t brn_bnn_workspace_bytes(int B, int P, int H, int C, int s_local);
/* Optional overlap of the minibatch copy with the sampling stage: `event` (cudaEvent_t, recorded by the caller on the
 * stream that copies X / y to the device) is waited for by the NEXT brn_bnn_elbo_fwd_bwd of this host thread immediately
 * before its first read of X and y -- noise generation and weight sampling run while the copy is in flight -- and is
 * then forgotten.  Replaces the host-side minibatch hand-over of EmpiricalDistribution._get_sample (distributions.py:410-462). */
void brn_set_data_ready_event(void* event);
int brn_bnn_elbo_fwd_bwd(const float* X, const int32_t* y, int B, int P, int H, int C,
                         const brn_mf_var vars[4], const brn_sample_range* r,
                         void* workspace, size_t workspace_bytes, int with_prior,
                         double* loss, void* stream);
/* The same with the hidden activation chosen: h = act(W1 x + b1), act in {tanh, relu, sigmoid} -- the link functions
 * BF.tanh / BF.relu / BF.sigmoid of brancher/functions.py:50-62 inside the BNN link.  brn_bnn_elbo_fwd_bwd == BRN_ACT_TANH. */
#define BRN_ACT_TANH 0
#define BRN_ACT_RELU 1
#define BRN_ACT_SIGMOID 2
int brn_bnn_elbo_fwd_bwd_act(const float* X, const int32_t* y, int B, int P, int H, int C, int activation,
                             const brn_mf_var vars[4], const brn_sample_range* r,
                             void* workspace, size_t workspace_bytes, int with_prior,
                             double* loss, void* stream);

/* K3 forward only -- batched posterior-predictive pass of the BNN (SURVEY 8(f)3): for S posterior weight samples and B data
 * rows, logits[s, b, :] = W2_s tanh(W1_s x_b + b1_s) + b2_s in one launch sequence (same sampler and tensor-core forward
 * GEMM as the ELBO evaluation), optionally labels[s, b] ~ Categorical(logits[s, b]) (Philox) and
 * probs_mean[b, c] += (1/S_total) softmax(logits[s, b])[c] (caller-zeroed).
 * Replaces ProbabilisticModel._get_posterior_sample (brancher/variables.py:796-812) as every evaluation loop of the examples
 * uses it -- one image and one graph walk at a time (tests/test_MNIST_bayesian_neural_network.py:75-81). */
int brn_bnn_predict(const float* X, int B, int P, int H, int C, int activation, const brn_mf_var vars[4],
                    const brn_sample_range* r, void* workspace, size_t workspace_bytes, float* logits, int32_t* labels,
                    float* probs_mean, void* stream);

/* K2 -- (multi-class) Bayesian logistic regression: logits_sbc = sum_f W_scf X_bf, W ~ q mean-field [C,F];
 *   likelihood 0: Bernoulli / Binomial(total_count=1, logits) with y float {0,1}  (C == 1)
 *   likelihood 1: Categorical(logits) with y int32 labels
 * over N observed rows (summed, variables.py:513-514).  Same accumulation contract as K3.
 * Replaces the graph walk for examples/minibatch_logistic_regression.py:27-43 /
 * examples/MNIST_logistic_regression.py (BF.matmul(weights, x) -> Binomial / Categorical). */
size_t brn_linear_workspace_bytes(int64_t N, int F, int C, int s_local);
int brn_linear_elbo_fwd_bwd(const float* X, const void* y, int likelihood, int64_t N, int F, int C,
                            const brn_mf_var* w, const brn_sample_range* r,
                            void* workspace, size_t workspace_bytes, int with_prior,
                            double* loss, void* stream);

/* K2 with a PREPARED data matrix.  The one-pass tcgen05 kernel (Bernoulli, C == 1, F a multiple of 16, F <= 128) reads X as a
 * power-of-two-scaled fp16 (hi, lo) pair.  brn_linear_elbo_fwd_bwd builds that pair on every call (one extra read of X for
 * the bound, one read + one write for the pair); an inference loop over a FIXED observed matrix -- the reference's
 * perform_inference over model.observe(data), brancher/inference.py:95-108 -- prepares it once and passes it to every
 * evaluation.  The caller owns `px` and must prepare it again whenever the contents of X change.
 *   brn_linear_prepared_x_bytes: size of the prepared form, 0 when it does not exist for this shape
 *   brn_linear_elbo_fwd_bwd_px:  px == NULL behaves exactly like brn_linear_elbo_fwd_bwd; a prepared X is ignored (X is
 *                                used) whenever the call does not take the one-pass kernel */
size_t brn_linear_prepared_x_bytes(int64_t N, int F);
int brn_linear_prepare_x(const float* X, int64_t N, int F, void* px, size_t px_bytes, void* stream);
int brn_linear_elbo_fwd_bwd_px(const float* X, const void* px, const void* y, int likelihood, int64_t N, int F, int C,
                               const brn_mf_var* w, const brn_sample_range* r,
                               void* workspace, size_t workspace_bytes, int with_prior,
                               double* loss, void* stream);

/* K2g -- Bayesian linear regression: y_b ~ Normal(sum_f w_sf X_bf, sigma_s) over N observed rows (summed, variables.py:513-514),
 * w ~ q mean-field [1, F] (`w`, Philox var_id 0 by convention).  Per sample, with r_sb = y_b - w_s . x_b and R_s = sum_b r_sb^2:
 *   ll_s = -R_s / (2 sigma_s^2) - N log sigma_s - N/2 log(2 pi) ;  loss += -(1/S_total) sum_{s local} ll_s
 * plus the prior / entropy terms of both latents (with_prior != 0; 0 drops them, for row-sharded callers).  Same accumulation
 * contract as K2.  Exactly one noise form is given:
 *   noise_scale != NULL: sigma_s = *noise_scale, a DEVICE fp32 scalar read on every call (a replayed CUDA graph sees a
 *                        re-assigned constant); nu must be NULL.
 *   nu != NULL:          sigma_s = nu_s, a scalar LogNormal latent (numel 1, Philox var_id 1 by convention):
 *                        q(nu) = LogNormal(mu, softplus(rho)), nu_s = exp(mu + softplus(rho) eps_s); the prior is
 *                        LogNormal(prior_loc, prior_scale), or q's own roots when tied.  log p(nu) = log N(log nu; a, b) - log nu
 *                        and H[q(nu)] = H[N(mu, softplus(rho))] + mu, as torch's LogNormal (TransformedDistribution) gives them.
 * y fp32 [N]; X fp32 [N, F], F <= 128; px: the prepared X of brn_linear_prepare_x, or NULL (used only when the call takes the
 * one-pass tensor-core kernel, as for brn_linear_elbo_fwd_bwd_px).  workspace: brn_linreg_workspace_bytes() bytes of scratch.
 * Replaces the graph walk of estimate_log_model_evidence (variables.py:843-870) for
 * NormalVariable(BF.matmul(weights, x), nu_or_constant, "y") -- examples/multivariate_regression.py with the regressors in a
 * matrix: _get_sample, _apply_link's batched matmul (variables.py:436-449), Normal / LogNormal log_prob and entropy
 * (distributions.py:111-124,170-181,493-507) and loss.backward() (inference.py:100). */
size_t brn_linreg_workspace_bytes(int64_t N, int F, int s_local);
int brn_linreg_elbo_fwd_bwd(const float* X, const void* px, const float* y, int64_t N, int F,
                            const brn_mf_var* w, const brn_mf_var* nu, const float* noise_scale,
                            const brn_sample_range* r, void* workspace, size_t workspace_bytes, int with_prior,
                            double* loss, void* stream);

/* K2g with a choice of likelihood: robust (heavy-tailed) regression over the same dense design matrix.  The codes continue the
 * likelihood codes of brn_linear_elbo_fwd_bwd (0 Bernoulli, 1 Categorical).  With r_sb = y_b - w_s . x_b, z_sb = r_sb / sigma_s
 * and u_s = log sigma_s, per sample (torch's log_prob of each distribution, summed over the N rows):
 *   BRN_LINREG_NORMAL   y_b ~ Normal(w_s . x_b, sigma_s):   ll_s = -sum_b r^2 / (2 sigma_s^2) - N u_s - N/2 log(2 pi)
 *                       exactly brn_linreg_elbo_fwd_bwd
 *   BRN_LINREG_CAUCHY   y_b ~ Cauchy(w_s . x_b, sigma_s):   ll_s = -N (log pi + u_s) - sum_b log1p(z^2)
 *   BRN_LINREG_LAPLACE  y_b ~ Laplace(w_s . x_b, sigma_s):  ll_s = -N (log 2 + u_s) - sum_b |r| / sigma_s
 *                       (the gradient of |r| at r = 0 is 0, as torch's abs gives it)
 * Every other argument, the two noise forms, the prior / entropy terms, the prepared X and the workspace are as for
 * brn_linreg_elbo_fwd_bwd.  Replaces the graph walk for CauchyVariable / LaplaceVariable(BF.matmul(weights, x), nu_or_constant,
 * "y") (standard_variables.py:156-183, torch.distributions Cauchy / Laplace log_prob). */
enum brn_linreg_likelihood { BRN_LINREG_NORMAL = 2, BRN_LINREG_CAUCHY = 3, BRN_LINREG_LAPLACE = 4 };
int brn_linreg_elbo_fwd_bwd_lik(const float* X, const void* px, const float* y, int likelihood, int64_t N, int F,
                                const brn_mf_var* w, const brn_mf_var* nu, const float* noise_scale,
                                const brn_sample_range* r, void* workspace, size_t workspace_bytes, int with_prior,
                                double* loss, void* stream);

/* K4a / K6b for regression: n weight vectors theta_k (or V_k) [n, F] at a FIXED noise scale, with ll_k the log-likelihood of
 * BRN_LINREG_NORMAL / _CAUCHY / _LAPLACE above (torch's log_prob summed over the N rows) at w_s = theta_k, sigma_s = *noise_scale.
 * The X pass is K2g's (the one-pass tensor-core kernel where the K2g evaluation of the same shape takes it, else the SIMT kernel)
 * with the vectors in place of the MC samples; a per-vector finisher replaces the mean-field one.  noise_scale: a DEVICE fp32
 * scalar, as for brn_linreg_elbo_fwd_bwd_lik; px: the prepared X of brn_linear_prepare_x, or NULL.  F <= 128; n == 0 and N == 0
 * are valid (N == 0: ll = 0).  workspace: brn_linreg_vectors_workspace_bytes() bytes of scratch.
 *   brn_linreg_particles_loss_grad:  loss += sum_k [ -ll_k - sum log N(theta_k; prior_loc, prior_scale) ]  (prior optional; a SUM
 *                                    over the particles, as brn_linear_particles_loss_grad), G = d loss / d theta (overwritten).
 *                                    Replaces SteinVariationalGradientDescent.compute_loss + loss.backward() (inference.py:292-299,
 *                                    100) and MAP's -log p(data, theta) + backward (inference.py:251-274) for
 *                                    Normal / Cauchy / LaplaceVariable(BF.matmul(weights, x), scale, "y").
 *   brn_linreg_vectors_loglik_grad:  ll[k] = ll_k (overwritten, fp64), G = -d ll_k / d V_k (overwritten) or G == NULL.
 *                                    Replaces the per-draw log-likelihoods of WassersteinVariationalGradientDescent.compute_loss
 *                                    (inference.py:203-229) for the same models; the rest of K6 is unchanged. */
size_t brn_linreg_vectors_workspace_bytes(int64_t N, int F, int n);
int brn_linreg_particles_loss_grad(const float* X, const void* px, const float* y, int likelihood, int64_t N, int F,
                                   const float* theta, int n, const float* prior_loc, const float* prior_scale,
                                   const float* noise_scale, float* G, double* loss,
                                   void* workspace, size_t workspace_bytes, void* stream);
int brn_linreg_vectors_loglik_grad(const float* X, const void* px, const float* y, int likelihood, int64_t N, int F,
                                   const float* V, int n, const float* noise_scale, float* G, double* ll,
                                   void* workspace, size_t workspace_bytes, void* stream);

/* K1 -- generic scalar-DAG ELBO: fused reparameterised sampling + log-probs + reduction over samples and data rows +
 * backward, for models whose variables are scalars (README.md:22-75 AR(1); examples/logNormal_normal.py;
 * examples/multivariate_regression.py).  The host flattens (joint, posterior) into a straight-line SSA program;
 * every op writes slot `dst` from slots a/b/c (or an immediate):
 *   leaves   CONST imm | PARAM params[a] | DATA data[row, a] | EPS standard normal of noise stream a for this sample
 *            (injected eps[s, a], or Philox(var_id = a, element 0))
 *   math     ADD SUB MUL DIV NEG POWI(imm) EXP LOG LOG1P SIGMOID SOFTPLUS(torch threshold 20) TANH SIN COS RELU SQRT ABS
 *            CLAMP_UNIT (torch SigmoidTransform's clamp to [tiny, 1-eps])
 *   density  NORMAL_LP(x=a, loc=b, scale=c) = torch Normal.log_prob ; NORMAL_ENTROPY(scale=a)
 *   reduce   ACC_SAMPLE a (latent log-prob / entropy term: once per sample) | ACC_ROW a (observed node: summed over
 *            the data axis, variables.py:513-514)
 *   loss += -(1/S_total) sum_{s local} [ sum ACC_SAMPLE + sum_rows ACC_ROW ] ; dparams[i] += d loss / d params[i].
 * LogNormal / LogitNormal sampling and densities are composed from these ops exactly in the order torch's
 * TransformedDistribution evaluates them (distributions.py:493-507 pattern).
 * Replaces the Python graph walk of estimate_log_model_evidence (variables.py:843-870, 486-570, 718-749) and
 * loss.backward() for this model class. */
enum brn_dag_opcode {
    BRN_DAG_CONST = 0, BRN_DAG_PARAM = 1, BRN_DAG_DATA = 2, BRN_DAG_EPS = 3,
    BRN_DAG_ADD = 4, BRN_DAG_SUB = 5, BRN_DAG_MUL = 6, BRN_DAG_DIV = 7, BRN_DAG_NEG = 8, BRN_DAG_POWI = 9,
    BRN_DAG_EXP = 10, BRN_DAG_LOG = 11, BRN_DAG_LOG1P = 12, BRN_DAG_SIGMOID = 13, BRN_DAG_SOFTPLUS = 14, BRN_DAG_TANH = 15,
    BRN_DAG_SIN = 16, BRN_DAG_COS = 17, BRN_DAG_RELU = 18, BRN_DAG_SQRT = 19, BRN_DAG_ABS = 20, BRN_DAG_CLAMP_UNIT = 21,
    BRN_DAG_NORMAL_LP = 22, BRN_DAG_NORMAL_ENTROPY = 23, BRN_DAG_ACC_SAMPLE = 24, BRN_DAG_ACC_ROW = 25,
    /* Optional layout markers (not operations).  A table may start with the sample-independent ("uniform") part of the
     * program -- ops that depend on parameters and constants only -- grouped by dependency level:
     *     UNIFORM_HEADER (a = number of entries that follow in the uniform segment,
     *                     b / c = number of EPS / DATA ops that lead the per-sample segment, in that order)
     *     { LEVEL (a = ops in this level, b = ops in the previous level) , ops of the level ... } *
     *     per-sample ops: EPS ops, DATA ops, then the rest in topological order
     * Bits 6 / 7 of a per-sample op's opcode fold an ACC_SAMPLE / ACC_ROW of its result into the op (opcodes are < 64).
     * The kernel evaluates the uniform segment once per CTA, the lanes of a warp taking the ops of a level in parallel,
     * instead of once per (sample, row) thread. */
    BRN_DAG_UNIFORM_HEADER = 26, BRN_DAG_LEVEL = 27
};
typedef struct brn_dag_op {
    int32_t opcode, dst, a, b, c;
    float   imm;
} brn_dag_op;
#define BRN_DAG_MAX_SLOTS 2048
#define BRN_DAG_MAX_PARAMS 2048
/* ops: DEVICE array [n_ops]; params/dparams [n_params]; data [n_rows, n_cols] (n_rows >= 1); eps [s_local, n_eps] or NULL */
int brn_dag_elbo_fwd_bwd(const brn_dag_op* ops, int n_ops, int n_slots, const float* params, int n_params,
                         const float* data, int n_cols, int n_rows, const float* eps, int n_eps,
                         const brn_sample_range* r, float* dparams, double* loss, void* stream);

/* Minibatch row indices drawn on the device, uniformly WITHOUT replacement: out [B] int64 holds B distinct values of
 * [0, N) in random order, a pure function of (N, B, seed, offset) (Philox4x32-10; duplicates are resolved by sequential-
 * rejection priority, see csrc/minibatch.cu).  Replaces np.random.choice(range(N), B, replace=False) of
 * EmpiricalDistribution._get_sample (distributions.py:410-462).  Requires B <= min(N / 2, 8192).
 * rounds (optional, device int): number of rejection rounds taken. */
int brn_minibatch_indices(int64_t N, int B, uint64_t seed, uint64_t offset, int64_t* out, int* rounds, void* stream);

/* K4 -- Stein variational gradient descent (SVGD).
 * (a) per-particle loss and gradient for (multi-class) logistic-regression particles theta [n, C*F]:
 *       loss += sum_k [ -sum_rows log-lik(theta_k) - sum log N(theta_k; prior_loc, prior_scale) ]     (prior optional)
 *       G[k]  = d loss / d theta_k                                                     (overwritten, [n, C*F])
 *     Replaces SteinVariationalGradientDescent.compute_loss + loss.backward() (inference.py:292-299, 100) for the
 *     model of development_playgrounds/SVGD_logistic_regression.py:34-48 (one ProbabilisticModel per particle).
 * (b) the SVGD direction for particles [row0, row0+rows) given ALL n particles and gradients (all-gathered by the
 *     host when particles are sharded over GPUs):
 *       D2_ij = ||theta_i - theta_j||^2 ; bw = 2 median_{i != j}(sqrt D2_ij)^2 / ln n   (exact np.median semantics)
 *       K_ij = exp(-D2_ij / (2 bw)) ; out_i = sum_j K_ij grad_j + (rowsum_i(K) theta_i - sum_j K_ij theta_j) / bw
 *     -- the reference's sign convention for the second term (attractive; canonical SVGD has the opposite sign) and
 *     no 1/n, exactly as SteinVariationalGradientDescent.correct_gradient / update_bandwidth compute it with four
 *     nested Python loops (inference.py:301-324).  `bandwidth` is a DEVICE float: written when update_bandwidth != 0,
 *     read otherwise.  out [rows, d] is overwritten. */
/*     workspace: brn_linear_particles_workspace_bytes() bytes of scratch selects the tcgen05 variant (the K2 GEMM pair
 *     with the particles as weight vectors; Bernoulli, C == 1, F % 4 == 0, large N and n); NULL / 0 runs the SIMT kernel. */
size_t brn_linear_particles_workspace_bytes(int64_t N, int F, int C, int n);
int brn_linear_particles_loss_grad(const float* X, const void* y, int likelihood, int64_t N, int F, int C,
                                   const float* theta, int n, const float* prior_loc, const float* prior_scale,
                                   float* G, double* loss, void* workspace, size_t workspace_bytes, void* stream);
size_t brn_svgd_workspace_bytes(int n, int d);
int brn_svgd_direction(const float* theta, const float* grad, int n, int d, int row0, int rows, int update_bandwidth,
                       float* bandwidth, float* out, void* workspace, size_t workspace_bytes, void* stream);

/* K4b sharded over ranks (one rank = a contiguous block of particle rows): the rank keeps only its rows of the distance
 * matrix, histograms its rows' part of the upper triangle, and the ranks ADD their histograms between the passes of the
 * exact median selection -- the one real exchange step of this path (brancher/inference.py:317-324 computes the median over
 * all pairs).  The collectives belong to the caller (NCCL through torch.distributed in the product); this entry runs the
 * device work between them, on the buffers whose byte offsets inside `workspace` brn_svgd_sharded_offsets reports:
 *   phase 0: D2 rows + level-0 histogram                       -> caller: all-reduce SUM of hist (4096 x uint32)
 *   phase 1, 2: scan of the previous level + next histogram    -> caller: all-reduce SUM of hist
 *   phase 3: last scan + successor pass                        -> caller: all-reduce SUM of cnt_le (uint64), MIN of next (uint32
 *                                                                 bit pattern of a non-negative float)
 *   phase 4: bandwidth (identical on every rank, bit for bit the replicated one) + update of the local rows -> out [rows, d]
 * theta, grad: ALL n particles (all-gathered by the caller).  Needs n % 4 == 0 and 8 <= d <= 143 (tensor-core kernels). */
size_t brn_svgd_sharded_workspace_bytes(int n, int d, int rows);
int brn_svgd_sharded_offsets(int n, int d, int rows, size_t* hist_off, size_t* hist_bytes, size_t* cnt_le_off, size_t* next_off);
int brn_svgd_sharded_phase(const float* theta, const float* grad, int n, int d, int row0, int rows, int phase,
                           float* bandwidth, float* out, void* workspace, size_t workspace_bytes, void* stream);

/* K5 -- amortised variational auto-encoder (examples/VAE_playground.py:30-80):
 *   encoder  h_0 = relu(W_0 x + b_0), ..., h_last ; mean = W_mean h_last + b_mean ; sd = softplus(W_sd h_last + b_sd) + sd_offset
 *   Qz = Normal(mean, sd) (amortised: its parameters are links, not roots), z = mean + sd*eps      (Normal.rsample)
 *   decoder  g_0 = relu(V_0 z + c_0), ..., g_last ; logits = V_out g_last + c_out ; x ~ Binomial(1, logits)
 *   p(z) = N(0, 1).  All weights are SHARED by the MC samples (nn.Module parameters, learnable_model=True,
 *   inference.py:129-139), so the contractions are ordinary [rows x features] GEMMs over rows = s_local * B.
 * Objective exactly as the reference evaluates it (SURVEY.md 8a'): x is not observed in p => no data-axis sum
 * (variables.py:513-514) => the estimator's .mean() runs over samples AND rows (gradient_estimators.py:44):
 *   loss += -(1/(s_total*B_total)) sum_{s local, b local} [ sum_pix (x l - log(1+e^l)) + sum_lat log N(z;0,1)
 *                                                           + sum_lat (1/2 + log sqrt(2 pi) + log sd_b) ]
 *           - log(s_total) * (add_constant != 0)      <- H[Qx] of EmpiricalDistribution._get_entropy (distributions.py:464-473)
 * and every layer's dW / db += d loss / d parameter (partials: rows [row0, row0+B) of B_total and samples
 * [s0, s0+s_local) of s_total; summing the partials of all ranks gives the full-batch result).
 * The SAME B rows are used by every MC sample (EmpiricalVariable(indices=...), distributions.py:443-455).
 * W layout = torch.nn.Linear.weight: [n_out][n_in] row-major.  X [B][D] fp32 in {0,1}.
 * eps: [s_local][B][L] injected noise or NULL -> Philox (element (row0+b)*L + l of stream var_id, global sample s).
 * Replaces the graph walk of estimate_log_model_evidence (variables.py:843-870) for this model: _get_sample with
 * BrancherFunction(nn.Module) links (functions.py:28-41, variables.py:436-449), Normal/Binomial log-probs
 * (distributions.py:476-490,561-575), analytic entropy (variables.py:156-162) and loss.backward() (inference.py:100). */
#define BRN_VAE_MAX_HIDDEN 6
typedef struct brn_dense_layer {
    const float* W;   /* [n_out][n_in] */
    const float* b;   /* [n_out]       */
    float*       dW;  /* += d loss / d W */
    float*       db;  /* += d loss / d b */
    int32_t      n_in, n_out;
} brn_dense_layer;
typedef struct brn_vae_model {
    int32_t D, L, n_enc, n_dec;        /* pixels, latent size, hidden layers of encoder / decoder (each >= 1) */
    float   sd_offset;                 /* 0.1 in the example */
    int32_t _pad;
    brn_dense_layer enc[BRN_VAE_MAX_HIDDEN];
    brn_dense_layer enc_mean, enc_sd;  /* heads: n_out = L */
    brn_dense_layer dec[BRN_VAE_MAX_HIDDEN];
    brn_dense_layer dec_out;           /* n_out = D */
} brn_vae_model;
size_t brn_vae_workspace_bytes(const brn_vae_model* m, int B, int s_local);
int brn_vae_elbo_fwd_bwd(const float* X, int B, int64_t row0, int64_t B_total, const brn_vae_model* m,
                         const float* eps, uint32_t var_id, const brn_sample_range* r,
                         void* workspace, size_t workspace_bytes, int add_constant, double* loss, void* stream);

/* K6 -- Wasserstein variational gradient descent (WassersteinVariationalGradientDescent, brancher/inference.py:154-248)
 * for ensembles of P (sampler, particle) pairs over one weight tensor of d = C*F elements -- the model class of
 * development_playgrounds/WVGD_logistic_regression.py:33-58: sampler k is q_k = N(loc_k, softplus(rho_k)), particle k a
 * learnable root theta_k.  One loss evaluation = three calls, each replacing P (or P^2) Python graph walks:
 * (a) brn_wvgd_sample_assign, once per noise draw (draw 0: sampler ELBOs, draw 1: particle loss; inference.py:203-212):
 *       Z[k,s,:] = loc_k + sigma_k * eps[k,s,:]              (eps injected, or Philox with var_id = 2k + draw -> eps_out)
 *       owner[k,s] = argmin_j cost(Z[k,s], theta_j)          (first minimal index)
 *     The truncation rule of sampler k accepts sample s iff owner[k,s] == k (inference.py:188-194; rejection with
 *     max_itr = 1, transformations.py:28-43 -- samples are masked, never compacted).  first_column_only != 0 reproduces
 *     the reference's numpy cost (utilities.py:125-126: only index 0 of the last axis, F_last elements apart, enters
 *     the squared distance); 0 = full squared distance.
 * (b) brn_linear_vectors_loglik_grad: ll[i] = sum_rows log-lik(data | weights = V[i]) and G[i] = -d ll[i] / d V[i] for
 *     n = P*S weight vectors in one fused pass over X (same kernel as K4a; G may be NULL).  Regression models (Normal / Cauchy /
 *     Laplace likelihood at a fixed noise scale) use brn_linreg_vectors_loglik_grad here instead.
 * (c) brn_wvgd_reduce: per sampler k, over its accepted samples A_k (draw 0) and A'_k (draw 1):
 *       loss += -mean_{A_k}[ll + log prior(z)]  +  sum_{A'_k} w_s ||theta_k - z'_s||^2
 *       w = softmax_{A'_k}(ll' + log prior(z') - log q_k(z'))   (1/S if biased)         (variables.py:821-841)
 *       dloc_k, drho_k: pathwise gradient of the first term (the entropy's detached-mean normaliser has no gradient:
 *       transformations.py:17-20 detaches the root samples as well); dtheta_k = 2 sum w_s (theta_k - z'_s).
 *     prior_loc == NULL: tied mode (p's auto-named roots take q_k's values, utilities.py:282-309).  A sampler with no
 *     accepted sample contributes nothing to the corresponding term (the reference re-draws until one is accepted);
 *     counts[k] = {|A_k|, |A'_k|}.  All outputs are overwritten except loss (+=). */
typedef struct brn_wvgd_args {
    const float *loc, *rho, *theta;          /* [P,d], [P,d] or [P] (rho_per_elem = 0), [P,d] */
    const float *prior_loc, *prior_scale;    /* [d] or NULL (tied) */
    const int32_t *owner0, *owner1;          /* [P,S] from (a), draws 0 and 1 */
    const double *ll0, *ll1;                 /* [P,S] from (b) */
    const float *G0;                         /* [P,S,d] from (b), draw 0 */
    const float *eps0, *eps1, *Z0, *Z1;      /* [P,S,d] */
    float *dloc, *drho, *dtheta;             /* [P,d] each (drho per element: sum it for a scalar rho) */
    int32_t *counts;                         /* [P,2] */
    double *loss;                            /* [1] += */
    int32_t P, S, d, rho_per_elem, biased, _pad;
} brn_wvgd_args;
int brn_wvgd_sample_assign(const float* loc, const float* rho, int rho_per_elem, const float* theta, const float* eps,
                           int P, int S, int d, int F_last, int first_column_only, int draw, const brn_sample_range* r,
                           float* Z, float* eps_out, int32_t* owner, void* stream);
int brn_linear_vectors_loglik_grad(const float* X, const void* y, int likelihood, int64_t N, int F, int C,
                                   const float* V, int n, float* G, double* ll, void* stream);
int brn_wvgd_reduce(const brn_wvgd_args* a, void* stream);

/* Tensor-core building block, exposed for validation: D[M][N] = A[M][K] . B[N][K]^T (all row-major fp32)
 * computed with tcgen05.mma kind::tf32 and the 3xTF32 hi/lo split (fp32-equivalent accuracy), TMA-fed.
 * This is the contraction the reference performs as a batched torch.matmul inside _apply_link
 * (variables.py:436-449 -> BF.matmul, functions.py:28-41). */
size_t brn_gemm_nt_workspace_bytes(int M, int N, int K);
int brn_gemm_nt_3xtf32(const float* A, const float* B, float* D, int M, int N, int K,
                       void* workspace, size_t workspace_bytes, void* stream);

/* ---- measurement hooks (bench.py): per-stage CUDA-event timing on the launch stream + launch count.
 * No reference counterpart (the reference has no profiler, SURVEY.md §5). */
void        brn_profile_enable(int on);
int         brn_profile_collect(void);                 /* synchronises the recorded events, sums them */
int         brn_profile_num_stages(void);
const char* brn_profile_stage(int i, double* total_ms, long long* calls);
void        brn_profile_reset(void);
long long   brn_launch_count(void);                    /* kernels launched by this library so far */

/* Fused optimiser step + loop bookkeeping without host synchronisation (SURVEY 8(f)1).
 * Replaces ProbabilisticOptimizer.update -> torch.optim.<name>.step() (brancher/optimizers.py:69-73) and, of the training
 * loop, the isfinite check / skip (brancher/inference.py:98,106-107) and the loss-curve bookkeeping (:105-109).
 * table_dev [n_tensors] and prefix_dev [n_tensors + 1] (first flat element index of each tensor; prefix[n] = total) live in
 * DEVICE memory.  counters_dev = int64[3]: {successful steps, iterations, skipped iterations}.  If *loss_dev is not finite
 * the parameters are left untouched.  curve_dev[iteration] = (float)*loss_dev when curve_dev != NULL and iteration <
 * curve_len.  *offset_dev (optional, see brn_sample_range.offset_dev) is incremented, so the next replay of a captured
 * iteration draws fresh Philox noise.
 * kind 0 = SGD (lr, momentum, weight_decay; dampening 0, no Nesterov), kind 1 = Adam (lr, beta1, beta2, eps, L2 weight_decay;
 * torch.optim.Adam's update, no amsgrad). */
typedef struct brn_opt_tensor {
    float* param;        /* [numel] updated in place                                   */
    const float* grad;   /* [numel]                                                     */
    float* m;            /* [numel] momentum buffer / Adam exp_avg (may be NULL for plain SGD) */
    float* v;            /* [numel] Adam exp_avg_sq (NULL for SGD)                      */
} brn_opt_tensor;
typedef struct brn_opt_hyper {
    int32_t kind; float lr, momentum, weight_decay, beta1, beta2, eps; int32_t _pad;
} brn_opt_hyper;
int brn_opt_step(const brn_opt_tensor* table_dev, const int64_t* prefix_dev, int n_tensors, int64_t total,
                 const brn_opt_hyper* hyper, const double* loss_dev, int64_t* counters_dev, float* curve_dev,
                 int64_t curve_len, uint64_t* offset_dev, void* stream);

/* One-shot all-reduce (sum) of a small fp32 buffer over peer memory (NVLink / NVSwitch), SURVEY 8e.  The reference has no
 * collective (single process, brancher/inference.py:50-111 runs on one device); this is the exchange step that finishes a
 * sample- / row-sharded evaluation: out[i] = sum_r src_r[i], summed in rank order on every rank (bit-identical results).
 * bufs_dev: DEVICE array [2 * world] of pointers, bufs[p * world + r] = rank r's symmetric buffer of parity p (n floats each,
 * 16-byte aligned, mapped into this process); flags_dev: DEVICE array [world], flags[r] = rank r's flag array (world
 * uint64, zero-initialised); state_dev: LOCAL device uint64[3], zero-initialised: {epoch, (ticket, time-out count), arrivals}; at most 16 ranks.
 * loss_inout (optional, device fp64 [1]): the partial loss travels in the buffer's LAST quad (elements n-4, n-3; needs
 * n % 4 == 0, the caller's src keeps that quad spare) as a (hi, lo) fp32 pair and is returned summed over ranks.
 * All ranks must issue the same sequence of calls (same n per state).  Enqueues ONE kernel; capturable in a CUDA graph. */
int brn_allreduce_oneshot(const float* src, float* out, int64_t n, float* const* bufs_dev,
                          unsigned long long* const* flags_dev, int rank, int world, uint64_t* state_dev,
                          double* loss_inout, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BRANCHER_CUDA_H */
