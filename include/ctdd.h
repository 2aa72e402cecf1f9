/*
 * ctdd.h — C ABI of libctdd_b200.so: B200 (sm_100a) kernels for the reverse-CTMC hot path of
 * continuous-time discrete diffusion (tauLDR / SDDM).
 *
 * The reference (paulffm/Continuous-Time-Diffusion-Models-for-Discrete-Data, "TAUnSDDM") is pure
 * PyTorch and has no FFI; each entry point below cites the reference Python code whose arithmetic it
 * replaces (paths relative to TAUnSDDM/).  The Python host classes in
 * continuous-time-diffusion-models-for-discrete-data_b200/lib/ bind these with ctypes.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (torch allocates); nothing is allocated,
 *     retained or freed by the library; all work is enqueued on `stream` (a cudaStream_t passed as
 *     void*) and is stream-ordered and re-entrant;
 *   - return value 0 = ok; non-zero = error, text available from ctdd_last_error() (thread-local);
 *   - matrices are row-major fp32; Q[k*S + s] = q_{t|0}(x_t = s | x_0 = k); Rb[i*S + j] = base rate
 *     of the forward jump i -> j (rows sum to 0); states are int32 in [0, S);
 *   - "row" means one (n, d) pair; rows are numbered n*D + d (+ row_offset for batch sharding).
 *     All randomness is counter-based Philox4x32-10 keyed on (seed, call offset, GLOBAL row), so results do
 *     not depend on the launch geometry or on the number of GPUs.  Tau-leap jump counts of a row are drawn
 *     through the Poisson superposition identity: total K ~ Poisson(sum_s lam_s), then K inverse-CDF picks
 *     over lam_s / sum (the same joint law as S independent Poisson draws; DESIGN.md §4.2, oracle/rng.py);
 *     with S <= 8 the uniform of K comes from a Philox call shared by 4 consecutive global rows.
 */
#ifndef CTDD_H_
#define CTDD_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CTDD_ABI_VERSION 1

/* ---- enums (plain ints in the ABI) ------------------------------------------------------------ */

/* how the reverse rates are formed from the logits */
enum {
  CTDD_BRANCH_TAULDR = 0,            /* lib/sampling/sampling.py:32-59  (CTElbo / NLL / CTElboLambda) */
  CTDD_BRANCH_SDDM_DIRECT = 1,       /* sampling.py:61-73 + lib/models/model_utils.py:38-39           */
  CTDD_BRANCH_SDDM_REVERSE_PROB = 2, /* model_utils.py:41-46                                          */
  CTDD_BRANCH_SDDM_REVERSE_LOGSCALE = 3 /* model_utils.py:49-54                                       */
};

/* what is done with the reverse rates */
enum {
  CTDD_MODE_TAU_LEAP = 0,        /* sampling.py:127-160 (TauL), :610-623 (PCTauL), :728-747 (Conditional) */
  CTDD_MODE_TAU_LEAP_CORR = 1,   /* sampling.py:170-221, :631-640: Poisson step on R_t[x,:] + rr          */
  CTDD_MODE_MIDPOINT_DRIFT = 2,  /* sampling.py:423-453: x' = clip(x + round(h/2 * sum_s rr_s (s-x)))     */
  CTDD_MODE_MIDPOINT_JUMP = 3,   /* sampling.py:459-503: rates at x_eval=x', jumps added to x_base=x      */
  CTDD_MODE_EULER = 4,           /* sampling.py:278-293 (LBJF)                                            */
  CTDD_MODE_EULER_CORR = 5,      /* sampling.py:296-341                                                   */
  CTDD_MODE_RATES_ONLY = 6,      /* get_reverse_rates only: writes rr_out / ratio_out, no state update    */
  CTDD_MODE_EXACT = 7            /* sampling.py:1008-1052 (ExactSampling): x' ~ Cat_s'( (softmax(logits) Q)[s'] * W[x][s'] );
                                    Q = q_{t-h|0}, and the RbT argument carries W[x][s'] = q_{t|t-h}[s', x]; branch, Rb,
                                    beta, h and eps are ignored; one per-row uniform (Euler stream)        */
};

/* which kernel family executes a reverse step */
enum {
  CTDD_IMPL_AUTO = 0,   /* S == 256 -> tcgen05 path, S <= 8 -> small-S path, else block path */
  CTDD_IMPL_SIMT = 1,   /* force the CUDA-core paths (used as on-GPU cross-check of the tensor path) */
  CTDD_IMPL_TC = 2      /* force the tcgen05 path (error if S != 256 or mode unsupported) */
};

/* stats_out layout (int64 counters, atomically incremented; caller zeroes) */
enum {
  CTDD_STAT_CHANGED_BASE = 0,  /* #rows with x_new != x_base           (TauL change_dim, sampling.py:161) */
  CTDD_STAT_NONZERO_JUMP = 1,  /* #rows whose unclamped jump sum != 0  (MidPointTauL change_dim, :505)    */
  CTDD_STAT_CHANGED_EVAL = 2,  /* #rows with x_new != x_eval           (MidPointTauL change_1to2, :506)   */
  CTDD_STAT_ROWS_JUMPED = 3,   /* #rows with sum_s k_s > 0             (:491)                             */
  CTDD_STAT_ROWS_MULTI = 4,    /* #rows with sum_s k_s > 1             (:493)                             */
  CTDD_STAT_COUNT = 8
};

/* ---- library ---------------------------------------------------------------------------------- */

int ctdd_version(void);
const char* ctdd_last_error(void);
/* number of kernels this library has launched in the calling process (bench.py's gpu_launches) */
long long ctdd_launch_count(void);

/* ---- q_{t|0} builders -------------------------------------------------------------------------
 * ctdd_build_qt0: Q_b = U diag(exp(lam * int_beta[b])) Uinv for b in [0,B); then, if `normalize`,
 * each row is divided by its sum; then entries < clamp_below are set to 0 (pass 0 to disable).
 * Replaces GaussianTargetRate.transition  lib/models/forward_model.py:265-287,
 *          UniformRate.transition         :108-126 (normalize=0, int_beta = t),
 *          UniformVariantRate.transit_between :180-200, BirthDeathForwardBase.transition :51-75
 *          (pass Uinv = U^T for the symmetric families).
 * Also writes, when non-null, QT (the transpose, [B,S,S]) — the layout the reverse-step kernels gather.
 */
int ctdd_build_qt0(const float* U, const float* Uinv, const float* lam, const float* int_beta,
                   int B, int S, int normalize, float clamp_below, float* Q_out, float* QT_out,
                   void* stream);

/* R_t scalar * base: out[b] = beta[b] * Rb   (forward_model.py:252-257, :166-172, :43-49) */
int ctdd_build_rate(const float* Rb, const float* beta, int B, int S, float* out, void* stream);

/* ---- reverse step -----------------------------------------------------------------------------
 * One reverse-rate evaluation over N*D rows fused with the state update selected by `mode`.
 * tauLDR branch (sampling.py:32-59):   ratio[s] = sum_k softmax(logits)[k] / (Q[k,x]+eps) * Q[k,s]
 *                                      rr[s]    = beta * Rb[s,x] * ratio[s]
 * SDDM branches (sampling.py:61-73):   ratio[s] = exp(ll[s] - ll[x]),  rr[s] = ratio[s] * beta * Rb[x,s]
 * The entry s == x is zeroed before any sampling (sampling.py:127-128, :423-427).
 */
typedef struct ctdd_step_params {
  int32_t mode;          /* CTDD_MODE_* */
  int32_t branch;        /* CTDD_BRANCH_* */
  int32_t impl;          /* CTDD_IMPL_* */
  int32_t N, D, S;
  int64_t row_offset;    /* global index of row 0 (batch sharding across GPUs) */
  const void* logits;    /* [N*D rows][S] of logits_dtype, row r at logits + r*ld_logits (elements) */
  int64_t ld_logits;     /* >= S, in elements of logits_dtype; lets a caller pass model output sliced as [:, cond:, :] */
  int64_t batch_stride_logits; /* elements of logits_dtype between consecutive n (= D_total*ld_logits for a sliced view, else D*ld_logits) */
  const int32_t* x_eval; /* [N*D] state the logits/rates were evaluated at */
  const int32_t* x_base; /* [N*D] state the jump is added to; NULL -> x_eval (only MIDPOINT_JUMP differs) */
  const float* Q;        /* [S,S] q_{t|0} at this step's time */
  const float* QT;       /* [S,S] transpose of Q */
  const float* Rb;       /* [S,S] base rate */
  const float* RbT;      /* [S,S] transpose of Rb */
  const void* tc_tables; /* blob from ctdd_prep_tc_tables for this time point, or NULL (SIMT only) */
  const void* tc_static; /* blob from ctdd_prep_tc_static (time-independent tables), or NULL (SIMT only) */
  float beta;            /* rate scalar beta(t) */
  float h;               /* step length (corrector multiplier already applied) */
  float eps;             /* sampler.eps_ratio */
  int32_t reject_multi;  /* 1: zero all jumps of a row whose jump count > 1 (not is_ordinal, sampling.py:135-138) */
  uint64_t seed;         /* Philox key */
  uint64_t offset;       /* Philox call counter (one per reverse-rate evaluation) */
  int32_t* x_out;        /* [N*D] new state (NULL allowed for RATES_ONLY) */
  float* rr_out;         /* [N*D,S] reverse rates incl. the (non-zeroed) s==x entry, or NULL */
  float* ratio_out;      /* [N*D,S] ratio, or NULL */
  int64_t* stats_out;    /* [CTDD_STAT_COUNT] or NULL */
  void* workspace;       /* >= ctdd_step_workspace_bytes(N*D, S) bytes, or NULL when that is 0 (it is 0 today) */
  /* Output head of the network (appended fields; zero-initialised = dense logits).  With CTDD_HEAD_LOGISTIC[_FIX] the
   * caller passes the two numbers per dimension the U-Net emits (lib/networks/unet.py:450-452) instead of the (N,D,S)
   * logits tensor and `logits` may be NULL: the kernel evaluates the truncated-logistic head
   * (lib/models/models.py:28-74, :248-282) on the fly, so the logits never exist in memory.  tcgen05 path (S == 256)
   * only; for other shapes materialise them with ctdd_logistic_logits first. */
  int32_t head;                 /* CTDD_HEAD_* */
  const void* head_mu;          /* of head_dtype; row (n,d) at head_mu[n*head_batch_stride + d] */
  const void* head_log_scale;   /* same type and addressing */
  int64_t head_batch_stride;    /* elements between consecutive n (2*D for the two halves of a torch.chunk'ed (B,2C,H,W)) */
  /* Element type of `logits` (appended field; zero-initialised = fp32): fp32, bf16 or fp16.  CTDD_DTYPE_BF16 and
   * CTDD_DTYPE_F16 take the logits a network run under torch.autocast (bf16 or its default fp16) emits without a widening
   * copy: the kernels widen on load (exact) and then run the fp32 arithmetic, so the states, counters, rr_out and
   * ratio_out equal those of the same call on the widened logits bit for bit.  The outputs stay fp32 / int32.  The
   * tcgen05 path (S == 256) needs 16-byte aligned rows: logits 16-byte aligned, ld_logits and batch_stride_logits
   * multiples of 8 elements for the 2-byte types (4 for fp32); a view that is not goes to the CUDA-core path under
   * CTDD_IMPL_AUTO and is refused under CTDD_IMPL_TC.  Ignored unless head == CTDD_HEAD_LOGITS. */
  int32_t logits_dtype;         /* CTDD_DTYPE_* */
  /* Element type of head_mu / head_log_scale (appended field; zero-initialised = fp32).  CTDD_DTYPE_BF16 takes the
   * (mu, log_scale) a U-Net run under torch.autocast(dtype=torch.bfloat16) emits without a widening copy: the kernels
   * widen on load (exact) and then run the fp32 head and step arithmetic, so the states, counters, rr_out and ratio_out
   * equal those of the same call on the widened (mu, log_scale) bit for bit.  fp32 or bf16 only: fp16 (mu, log_scale)
   * are O(N*D) and are widened by the caller.  Ignored when head == CTDD_HEAD_LOGITS; otherwise any other value is
   * refused with status 2 before any CUDA call. */
  int32_t head_dtype;           /* CTDD_DTYPE_* */
} ctdd_step_params;

enum {
  CTDD_DTYPE_F32 = 0,          /* float32 logits */
  CTDD_DTYPE_BF16 = 1,         /* bfloat16 logits */
  CTDD_DTYPE_F16 = 2           /* float16 (IEEE half) logits */
};

enum {
  CTDD_HEAD_LOGITS = 0,        /* dense logits */
  CTDD_HEAD_LOGISTIC = 1,      /* model.model_output == 'logistic_pars', fix_logistic False */
  CTDD_HEAD_LOGISTIC_FIX = 2   /* fix_logistic True: min with the mirrored evaluation (models.py:66-70) */
};

/* logits[n,d,s] of the truncated-logistic head: log-mass of Logistic(mu, exp(log_scale - 2)) on bin s of [-1,1] cut into
 * S bins, with the reference's 1e-6 guard.  Replaces sample_logistic lib/models/models.py:28-74 (one pass instead of ~20
 * elementwise passes over (N,D,S)).  Values agree with the reference to its own fp32 noise; see DESIGN.md. */
int ctdd_logistic_logits(const float* mu, const float* log_scale, int N, int D, int64_t batch_stride, int S,
                         int fix_logistic, float* logits_out, void* stream);
/* Backward of the head w.r.t. its two inputs: grad_mu[n,d] = sum_s grad_logits[n,d,s] * dlogits/dmu (same for log_scale),
 * written at the addressing of mu / log_scale.  Replaces autograd through the ~20 saved (N,D,S) tensors of the
 * reference's formula chain (models.py:44-72); recomputes the head from (mu, log_scale), reads grad_logits once. */
int ctdd_logistic_logits_backward(const float* mu, const float* log_scale, const float* grad_logits, int N, int D,
                                  int64_t batch_stride, int S, int fix_logistic, float* grad_mu, float* grad_log_scale,
                                  void* stream);
/* The two calls above with explicit element types (the calls above are these with fp32 everywhere).  in_dtype (mu /
 * log_scale) is CTDD_DTYPE_F32 or CTDD_DTYPE_BF16; out_dtype (logits_out) and grad_dtype (grad_logits) are
 * CTDD_DTYPE_F32, CTDD_DTYPE_BF16 or CTDD_DTYPE_F16.  2-byte inputs are widened on load (exact) and the fp32 arithmetic
 * runs unchanged:
 *   - ctdd_logistic_logits_ex: fp32 logits_out equal those of the fp32 call on the widened inputs bit for bit; bf16 and
 *     fp16 logits_out are those values rounded once, to nearest even (fp16: overflow gives +-inf, small values become
 *     subnormals).  Four logits are stored at once when S % 4 == 0 and logits_out is aligned to 4 elements (16 bytes
 *     fp32, 8 bytes for the 2-byte types), one at a time otherwise;
 *   - ctdd_logistic_logits_backward_ex: grad_mu / grad_log_scale stay fp32 (at the addressing of mu) and equal those of
 *     the fp32 call on the widened tensors bit for bit, provided grad_logits is aligned to 4 of its elements whenever the
 *     widened copy is 16-byte aligned (the accumulation order depends on that alignment, not on the type).
 * Any other dtype is refused with status 2 before any launch. */
int ctdd_logistic_logits_ex(const void* mu, const void* log_scale, int in_dtype, int N, int D, int64_t batch_stride, int S,
                            int fix_logistic, void* logits_out, int out_dtype, void* stream);
int ctdd_logistic_logits_backward_ex(const void* mu, const void* log_scale, int in_dtype, const void* grad_logits,
                                     int grad_dtype, int N, int D, int64_t batch_stride, int S, int fix_logistic,
                                     float* grad_mu, float* grad_log_scale, void* stream);

int64_t ctdd_step_workspace_bytes(int64_t rows, int S, int impl);
int ctdd_reverse_step(const ctdd_step_params* p, void* stream);

/* Derived per-time-point tables for the tcgen05 path (S == 256): bf16 hi/mid splits of Q^T in the
 * order the kernel loads them into tensor memory and the gathered-denominator table 1/(Q[k,x]+eps)
 * (tauLDR; Q[k,x] for the SDDM branch).  T time points at once.  The tables depend on QT, eps and
 * branch only: Q and Rb are not read (either may be NULL). */
int64_t ctdd_tc_tables_bytes(int S);
/* time-independent tables of the tcgen05 path: Rb^T and Rb with zeroed and with kept diagonals (epilogue gathers), a zero
 * row, the band of non-zero base rates per state.  static_out must be aligned to ctdd_tc_static_align() bytes
 * (the epilogue addresses the blob with 32-bit offsets under a constant upper address word). */
int64_t ctdd_tc_static_bytes(int S);
int64_t ctdd_tc_static_align(void);
int ctdd_prep_tc_static(const float* Rb, int S, void* static_out, void* stream);
int ctdd_prep_tc_tables(const float* Q, const float* QT, const float* Rb, int T, int S, float eps,
                        int branch, void* tables_out, void* stream);

/* ---- initial / forward-noising samplers ------------------------------------------------------- */

/* x[r] ~ Categorical(prob[0..S)) by inverse CDF on one Philox uniform per row.
 * Replaces get_initial_samples  lib/sampling/sampling.py:14-28 (uniform: prob = 1/S). */
int ctdd_sample_categorical_shared(const float* prob, int S, int64_t rows, int64_t row_offset,
                                   uint64_t seed, uint64_t offset, int32_t* x_out, void* stream);

/* x_t[b,d] ~ Categorical(Q[b, x0[b,d], :])      lib/losses/losses.py:46-59 (and :326-338, :862-874)
 * then x~: one dimension d* ~ Cat(sum_{s!=x_t} R[b,x_t[d],s]) and a new value ~ Cat(R[b,x_t[d*],.] off-diag)
 *                                                 lib/losses/losses.py:61-101.
 * Q: [B,S,S]; Rb: [S,S]; beta: [B]; x_tilde_out may be NULL (CatRM family needs only x_t). */
int ctdd_noise_xt(const float* Q, const float* Rb, const float* beta, const int32_t* x0, int B, int D,
                  int S, int64_t batch_offset, uint64_t seed, uint64_t offset, int32_t* xt_out,
                  int32_t* x_tilde_out, void* stream);

/* ---- training-step plumbing --------------------------------------------------------------------
 * EMA of the model parameters, every trainable tensor in one launch:
 *   shadow <- shadow - one_minus_decay * (shadow - param)        EMA.update_ema  lib/models/models.py:745-758
 * (the reference loops over the parameters in Python).  chunk_table: device array of n_chunks records
 * {float* shadow; const float* param; int64_t n;} (24 bytes each), a tensor cut into pieces of at most
 * ctdd_ema_chunk_elems() elements.  Same roundings as the reference's torch expression (bitwise equal results). */
#define CTDD_EMA_CHUNK 32768
int64_t ctdd_ema_chunk_elems(void);
int ctdd_ema_update(const void* chunk_table, int n_chunks, float one_minus_decay, void* stream);

/* ---- evaluation metrics (SURVEY §8f-4) ------------------------------------------------------------
 * Pair similarities of two sample sets X (N, D), Y (M, D), fp32 row-major (the reference casts to float32 first):
 *   k(x, y) = exp(-bd * sum_d |x_d - y_d|)      binary_exp_hamming_sim  lib/datasets/metrics.py:14-22, lib/utils/utils.py:101-105
 *   k(x, y) = D - sum_d |x_d - y_d|             binary_hamming_sim      lib/datasets/metrics.py:6-10     (hamming_sim != 0)
 * ctdd_pair_similarity writes the (N, M) matrix K.  ctdd_pair_similarity_sum writes ONE double to `out`: the sum of k
 * over all pairs, or with self != 0 (needs X == Y, N == M) over the pairs i != j — the three sums of binary_mmd
 * (metrics.py:25-48) without the (N, M, D) difference tensor.  `partials` is caller scratch of ctdd_pair_partials(N, M)
 * doubles; the reduction order is fixed (deterministic).  N == 0 or M == 0 gives 0. */
int64_t ctdd_pair_partials(int N, int M);
int ctdd_pair_similarity(const float* X, int N, const float* Y, int M, int D, float bd, int hamming_sim, float* K, void* stream);
int ctdd_pair_similarity_sum(const float* X, int N, const float* Y, int M, int D, float bd, int self, int hamming_sim,
                             double* partials, double* out, void* stream);
/* Per-dimension state counts of a sample set x (N, D) int32: counts[d*S + s] += #{n : x[n,d] == s}; counts has D*S + 1
 * entries, the last one counts out-of-range states (a correct sampler leaves it 0).  The caller zeroes counts; successive
 * calls accumulate (batch sharding).  S <= 8192.  Used for the per-dimension histogram / KL check of the reverse process. */
int ctdd_state_histogram(const int32_t* x, int64_t N, int D, int S, int32_t* counts, void* stream);

/* ---- loss terms -------------------------------------------------------------------------------
 * All per-sample reductions are returned as [B] vectors; the (tiny) final means/weights are combined by
 * the Python loss classes exactly as lib/losses/losses.py does, so one kernel serves every loss class.
 */
typedef struct ctdd_loss_params {
  int32_t kind;          /* CTDD_LOSS_* */
  int32_t logit_type;    /* CTDD_BRANCH_SDDM_* (CRM / SDDM kinds) */
  int32_t crm_type;      /* 0 rm, 1 mle, 2 elbo (loss.loss_type, losses.py:794-836) */
  int32_t B, D, S;
  const void* logits;    /* [B,D,S] of logits_dtype */
  const float* Q;        /* [B,S,S] */
  const float* QT;       /* [B,S,S] */
  const float* Rb;       /* [S,S] */
  const float* beta;     /* [B] */
  const int32_t* x0;     /* [B,D] minibatch */
  const int32_t* xt;     /* [B,D] state the reg / ratio terms are evaluated at (CTELBO: reg_x; SDDM, CRM: state of the logits) */
  const int32_t* x_tilde;/* [B,D] CTELBO: state of the signal term; SDDM: NULL (== xt); CRM: unused */
  float eps;
  /* forward outputs, per sample [B]; the caller zeroes them (the kernel accumulates with atomics) */
  float* out_a;          /* CTELBO / SDDM: reg term                       CRM: sum_d loss_type term */
  float* out_b;          /* CTELBO / SDDM: outer_sum (signal)                                      */
  float* out_c;          /* CTELBO / SDDM: sig_norm (does not depend on the logits)                */
  float* out_d;          /* SDDM / CRM: sum_d (-ll_x)   (ScoreElbo's ratio-matching term)          */
  float* out_nll;        /* sum_d CrossEntropy(logits[b,d,:], x0[b,d])                            */
  /* backward: grad_logits[b] = ga[b]*d out_a + gb[b]*d out_b + gd[b]*d out_d + gn[b]*d out_nll */
  const float* ga; const float* gb; const float* gd; const float* gn;
  void* grad_logits;     /* [B,D,S] of logits_dtype (bf16 / fp16 logits get a bf16 / fp16 gradient) */
  void* workspace;       /* >= ctdd_loss_workspace_bytes(kind, B, S); written by forward, read by backward */
  /* appended field (zero-initialised = CUDA-core contractions).  S == 256, kinds SDDM and CRM with reverse_prob /
   * reverse_logscale: >= ctdd_loss_tc_scratch_bytes(B, D, S) bytes, 16-byte aligned; the two (B*D x S)(S x S) contractions
   * then run on tcgen05 (ctdd_bgemm256_tc).  Written by forward, read AND overwritten by backward: pass the same buffer to
   * both calls, untouched in between.  Ignored for CT-ELBO and the `direct` logit type. */
  void* tc_scratch;
  /* Element type of `logits` and `grad_logits` (appended field; zero-initialised = fp32): CTDD_DTYPE_F32,
   * CTDD_DTYPE_BF16 or CTDD_DTYPE_F16, as in ctdd_step_params.  bf16 and fp16 take the logits a network run under
   * torch.autocast (bf16 or its default fp16) emits without a widening copy: the kernels widen on load (exact), run the
   * fp32 arithmetic, and round the gradient once (to nearest even) when they store it.  The per-sample outputs equal
   * those of the same call on the widened logits up to the order of the per-CTA atomicAdds, and grad_logits equals that
   * call's fp32 gradient rounded to the logits' type, bit for bit (fp16: overflow gives +-inf, as a loss scaler expects).
   * The outputs, ga..gn, workspace and tc_scratch stay fp32.  On the tensor-core path (tc_scratch at S == 256) logits and
   * grad_logits must be 16-byte aligned for every type; other pointers are refused with status 2 before any launch. */
  int32_t logits_dtype;  /* CTDD_DTYPE_* */
} ctdd_loss_params;

enum {
  CTDD_LOSS_CTELBO = 0,  /* lib/losses/losses.py:108-286 (CTElbo, NLL, CTElboLambda; one_forward_pass) */
  CTDD_LOSS_CRM = 1,     /* losses.py:794-890 (CatRM, CatRMNLL) */
  CTDD_LOSS_SDDM = 2     /* losses.py:1345-1500 (ScoreElbo), :389-544 (SDDMElbo) */
};

/* Per-sample contraction of the loss terms on tcgen05 (S == 256 only): out[b,d,n] = sum_k X[b,d,k] * M[b,n,k], fp32 in / out,
 * 3 x BF16 split precision (relative error ~3e-5).  Replaces the batched matmuls with a per-sample q_{t|0} of
 * lib/losses/losses.py:148-150, :179-181 and lib/models/model_utils.py:44-46 (forward: M = QT, backward: M = Q).
 * X, out: [B, D, 256]; M: [B, 256, 256]; all 16-byte aligned. */
int ctdd_bgemm256_tc(const float* X, const float* M, int B, int D, float* out, void* stream);

int64_t ctdd_loss_workspace_bytes(int kind, int B, int S);
int64_t ctdd_loss_tc_scratch_bytes(int B, int D, int S);
int ctdd_loss_forward(const ctdd_loss_params* p, void* stream);
int ctdd_loss_backward(const ctdd_loss_params* p, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CTDD_H_ */
