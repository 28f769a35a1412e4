/*
 * pilco_b200.h -- C ABI of the B200-native PILCO moment-matching rollout engine.
 *
 * The reference (nrontsis/PILCO) has no FFI: its hot path is TensorFlow ops composed in Python.
 * This ABI is therefore the boundary placed directly beneath the reference's Python class API;
 * each entry point names the reference function (file:line under /root/reference) it replaces.
 *
 * Rules (all entry points):
 *   - every pointer is a DEVICE pointer to contiguous fp64 (or int32 for `info`), owned by the caller
 *     (PyTorch allocates them); the library never allocates or frees device memory;
 *   - work is only enqueued on the `stream` argument; no entry point synchronises the device
 *     (so every `*_forward/_backward/rollout` call is CUDA-graph capturable);
 *   - return value: 0 ok, <0 invalid argument (see pilco_status_string); numerical failures
 *     (non-PD matrices) are reported per batch element in the device `info` array
 *     (0 ok, bit0: non-PD input-covariance system, bit1: non-PD Gram matrix);
 *   - batch dimension R = independent rollouts ("policy restarts", pilco/models/pilco.py:98-107);
 *   - matrices are row-major; `*_bs` arguments are batch strides in doubles (0 = one array shared
 *     by all R batch elements).
 */
#ifndef PILCO_B200_H
#define PILCO_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PILCO_ABI_VERSION 3
#define PILCO_MAX_D 16          /* max GP input dimension (state+control) */
#define PILCO_MAX_E 16          /* max number of GP outputs */

typedef void* pilco_stream_t;   /* cudaStream_t */

/* ---- ABI / sizing ------------------------------------------------------------------------- */
int         pilco_version(void);
const char* pilco_status_string(int status);
/* rows/cols of every per-centre array are padded to a multiple of 64 */
int         pilco_pad_n(int n);
/* workspace bytes for pilco_mm_forward / pilco_mm_backward with these sizes */
size_t      pilco_mm_workspace_bytes(int n, int D, int E, int R);

/* ---- moment matching ------------------------------------------------------------------------
 * Replaces MGPR.predict_given_factorizations (pilco/models/mgpr.py:91-149; MATLAB gp0.m:63-104,
 * gp1.m:85-124, gp2.m:69-106): Gaussian input N(m,s) -> predictive mean M, covariance S and
 * V = inv(s) * input-output covariance, for E independent SE-ARD GPs over n centres.
 */
typedef struct pilco_gp_model {
    int n, D, E;
    int mode;               /* 0: GP with trace term, +sf2 on diag(S) (mgpr.py:143-147);
                               1: deterministic GP / RBF network: no trace term, +1e-6
                                  (controllers.py:116-117, gp2.m:96-99) */
    const double* X;    long long X_bs;     /* [n,D] centres (training inputs / inducing points / RBF centres) */
    const double* ell;  long long ell_bs;   /* [E,D] lengthscales */
    const double* sf2;  long long sf2_bs;   /* [E] signal variances */
    const double* beta; long long beta_bs;  /* [E,n] (K+sn2 I)^-1 y */
    const double* iK;   int ldk;            /* [E,ldk,ldk] (K+sn2 I)^-1, zero padded, ldk >= pilco_pad_n(n);
                                               NULL when mode==1.  Shared by the batch. */
} pilco_gp_model;

int pilco_mm_forward(const pilco_gp_model* gp, int R,
                     const double* m,       /* [R,D]   */
                     const double* s,       /* [R,D,D] */
                     double* M,             /* [R,E]   */
                     double* S,             /* [R,E,E] */
                     double* V,             /* [R,D,E] */
                     int* info,             /* [R] or NULL */
                     void* ws, size_t ws_bytes, pilco_stream_t stream);

/* VJP of pilco_mm_forward (the reference differentiates mgpr.py:91-149 with TensorFlow autodiff inside
 * gpflow.optimizers.Scipy, pilco/models/pilco.py:84-90).  Inputs: the forward inputs m, s, the forward output
 * M and the cotangents gM [R,E], gS [R,E,E], gV [R,D,E].  Outputs gm [R,D], gs [R,D,D] (symmetric part) and,
 * when all three pointers are non-NULL (trainable RBF policy), gX [R,n,D], gbeta [R,E,n], gell [R,E,D]. */
size_t pilco_mm_bwd_workspace_bytes(int n, int D, int E, int R, int need_param);
int pilco_mm_backward(const pilco_gp_model* gp, int R, const double* m, const double* s, const double* M,
                      const double* gM, const double* gS, const double* gV,
                      double* gm, double* gs, double* gX, double* gbeta, double* gell,
                      void* ws, size_t ws_bytes, pilco_stream_t stream);

/* Taped moment match: pilco_mm_forward that also leaves, per unordered output pair (a,b), the row sums, column sums
 * and the product (G_ab o L'_ab) Z of the N x N matrix it has in registers anyway (Z = centred inputs) on a tape;
 * pilco_mm_backward_taped turns the tape and the cotangents into gm, gs WITHOUT recomputing an exponential.
 * Only the cotangents of the input moments are produced (the dynamics GP of the policy objective, whose inputs
 * and hyper-parameters are constants, pilco/models/pilco.py:80-82); trainable centres need pilco_mm_backward. */
size_t pilco_mm_tape_bytes(int n, int D, int E, int R);          /* 0: shape not supported (n > 1024 for D <= 12, n > 704 beyond) */
size_t pilco_mm_tape_bwd_workspace_bytes(int D, int E, int R);
int pilco_mm_forward_taped(const pilco_gp_model* gp, int R, const double* m, const double* s,
                           double* M, double* S, double* V, int* info,
                           void* ws, size_t ws_bytes, void* tape, size_t tape_bytes, pilco_stream_t stream);
int pilco_mm_backward_taped(const pilco_gp_model* gp, int R, const double* m, const double* s, const double* M,
                            const double* gM, const double* gS, const double* gV,
                            const void* tape, size_t tape_bytes, double* gm, double* gs,
                            void* ws, size_t ws_bytes, pilco_stream_t stream);

/* ---- GP factorisation -----------------------------------------------------------------------
 * Replaces MGPR.calculate_factorizations (pilco/models/mgpr.py:81-89; gp0.m:46-61):
 * K_e = sf2_e exp(-0.5 |(x-x')/ell_e|^2); L = chol(K + sn2_e I); iK = (K+sn2 I)^-1; beta = iK y_e.
 * B batch elements (B=1 for the dynamics GP; B=R for per-restart RBF policies).
 * iK is written with leading dimension ldk (zero padded; pass NULL to get beta only).
 * ws: scratch of pilco_gp_factorize_workspace_bytes(n, E, B) bytes; on return its first
 * B*E*ldw*ldw doubles (ldw = pilco_pad_n(n)) hold the Cholesky factors L (lower triangles), which
 * pilco_rollout_backward needs for the RBF policy (pilco_rollout_grad.pol_L).
 */
size_t pilco_gp_factorize_workspace_bytes(int n, int E, int B);
int pilco_gp_factorize(int n, int D, int E, int B,
                       const double* X,   long long X_bs,    /* [n,D]  */
                       const double* Y,   long long Y_bs,    /* [n,E]  */
                       const double* ell, long long ell_bs,  /* [E,D]  */
                       const double* sf2, long long sf2_bs,  /* [E]    */
                       const double* sn2, long long sn2_bs,  /* [E]    */
                       double* iK, int ldk,                  /* [B,E,ldk,ldk] or NULL */
                       double* beta,                         /* [B,E,n] */
                       int* info,                            /* [B] or NULL */
                       void* ws, size_t ws_bytes, pilco_stream_t stream);

/* Incremental set_data (SURVEY section 8f-2): k rows appended to the data of a factorised model with UNCHANGED
 * hyper-parameters (pilco/models/mgpr.py:38-45; examples/inv_double_pendulum.py:102-103, swimmer.py:87-88 append the
 * rows of each new episode).  X [n0+k, D] and Y [n0+k, E] hold the old rows first; iK_old [E,ldk_old,ldk_old] is the
 * inverse pilco_gp_factorize / an earlier append produced.  Writes the new zero-padded inverse iK_new
 * [E,ldk_new,ldk_new] (ldk_new >= pilco_pad_n(n0+k), out of place) and beta_new [E,n0+k] by the block-inverse
 * (Schur complement) update: O(n^2 k) instead of O(n^3).  info[0] bit 1: Schur complement not positive definite. */
size_t pilco_gp_append_workspace_bytes(int n0, int k, int E);
int pilco_gp_append(int n0, int k, int D, int E,
                    const double* X, const double* Y,
                    const double* ell, const double* sf2, const double* sn2,
                    const double* iK_old, int ldk_old,
                    double* iK_new, int ldk_new, double* beta_new, int* info,
                    void* ws, size_t ws_bytes, pilco_stream_t stream);

/* GP training objective (SURVEY section 8f-1): nlml[b,e] = -log p(y_e | X, theta_be) and its gradient w.r.t. the
 * constrained hyper-parameters, batched over B hyper-parameter sets x E outputs.  Replaces
 * gpflow.models.GPR.training_loss + TF autodiff inside MGPR.optimize (pilco/models/mgpr.py:47-75); the Gamma priors
 * of mgpr.py:33-34 are added by the host.  Outputs nlml [B,E], g_ell [B,E,D], g_sf2 [B,E], g_sn2 [B,E]. */
size_t pilco_gp_nlml_workspace_bytes(int n, int E, int B);
int pilco_gp_nlml(int n, int D, int E, int B,
                  const double* X,   long long X_bs, const double* Y,   long long Y_bs,
                  const double* ell, long long ell_bs, const double* sf2, long long sf2_bs,
                  const double* sn2, long long sn2_bs,
                  double* nlml, double* g_ell, double* g_sf2, double* g_sn2, int* info,
                  void* ws, size_t ws_bytes, pilco_stream_t stream);

/* FITC training objective (SURVEY section 8f-1, sparse half): value and gradient of the collapsed FITC bound
 * (gpflow.models.GPRFITC.training_loss as SMGPR.optimize minimises it, pilco/models/smgpr.py:16-22 via
 * mgpr.py:47-75; no priors) w.r.t. the constrained hyper-parameters AND the inducing inputs, batched over B
 * parameter sets x E outputs -- every output trains its own Z [Mi,D].  X [N,D], Y [N,E] are shared by the batch;
 * Z [B,E,Mi,D], ell [B,E,D], sf2/sn2 [B,E].  Outputs nlml [B,E], g_ell [B,E,D], g_sf2, g_sn2 [B,E], g_Z [B,E,Mi,D].
 * info[b] bit 1: a Cholesky factorisation (Kuu + 1e-6 I, or I + V diag(1/nu) V') failed. */
size_t pilco_fitc_nlml_workspace_bytes(int N, int Mi, int D, int E, int B);
int pilco_fitc_nlml(int N, int Mi, int D, int E, int B,
                    const double* X, const double* Y, const double* Z,
                    const double* ell, const double* sf2, const double* sn2,
                    double* nlml, double* g_ell, double* g_sf2, double* g_sn2, double* g_Z, int* info,
                    void* ws, size_t ws_bytes, pilco_stream_t stream);

/* Replaces SMGPR.calculate_factorizations (pilco/models/smgpr.py:24-45; gp1.m:52-82): FITC over
 * Mi inducing points Z.  Outputs iK[E,ldk,ldk] (zero padded) and beta[E,Mi].
 * ws: scratch of pilco_fitc_workspace_bytes(N, Mi, E) bytes. */
size_t pilco_fitc_workspace_bytes(int N, int Mi, int E);
int pilco_fitc_factorize(int N, int Mi, int D, int E,
                         const double* X,   /* [N,D]  */
                         const double* Z,   /* [Mi,D] */
                         const double* Y,   /* [N,E]  */
                         const double* ell, const double* sf2, const double* sn2,
                         double* iK, int ldk, double* beta,
                         int* info, void* ws, size_t ws_bytes, pilco_stream_t stream);

/* ---- prediction at deterministic inputs -------------------------------------------------------
 * Replaces gpflow.models.GPR.predict_f / GPRFITC.predict_f, the methods users call on pilco.mgpr.models[i]
 * (pilco/models/mgpr.py:28-36, smgpr.py:16-22; examples/"Hyperparameter setting and troubleshooting tips.ipynb",
 * "Check the one-step predictions manually"), and through them predict_y / predict_log_density.  For B test points
 * Xs and every output e, from the factors pilco_gp_factorize / pilco_fitc_factorize / pilco_gp_append leave (mode 0):
 *   mean[b,e] = k*' beta_e,   var[b,e] = sf2_e - k*' iK_e k*   (latent, no noise),   k* = k_e(centres, Xs[b])
 *   cov[e]    = K_e(Xs, Xs) - K*' iK_e K*                          (full_cov)
 * Any of mean / var / cov may be NULL (not all three); var and cov need gp->iK.  The diagonal path is one fused kernel that
 * never writes K* to memory and needs no workspace (pilco_gp_predict_workspace_bytes(..., 0) == 0); a point's result is
 * bitwise independent of B and of its position in the batch.  cov needs 2 E B pad_n(n) doubles of workspace.
 * gp must be unbatched (all *_bs == 0); one output i of an E-output model is predicted by passing E = 1 with ell, sf2,
 * beta and iK offset to output i.  B == 0 is a no-op.  PILCO_ERR_UNSUPPORTED: n > 3472 centres. */
size_t pilco_gp_predict_workspace_bytes(int n, int D, int E, int B, int full_cov);
int    pilco_gp_predict(const pilco_gp_model* gp, int B, const double* Xs /*[B,D]*/,
                        double* mean /*[B,E] or NULL*/, double* var /*[B,E] or NULL*/,
                        double* cov /*[E,B,B] or NULL*/, void* ws, size_t ws_bytes, pilco_stream_t stream);

/* ---- closed-form moments ---------------------------------------------------------------------
 * squash_sin (pilco/controllers.py:13-36; gSin.m:33-48), LinearController.compute_action
 * (controllers.py:46-58; conlin.m:50-62), ExponentialReward.compute_reward (rewards.py:19-51;
 * reward.m:35-57).  All batched over R.
 */
int pilco_squash_sin(int U, int R, const double* m /*[R,U]*/, const double* s /*[R,U,U]*/,
                     const double* max_action /*[U]*/,
                     double* M /*[R,U]*/, double* S /*[R,U,U]*/, double* C /*[R,U,U]*/,
                     pilco_stream_t stream);

int pilco_linear_action(int Ds, int U, int R,
                        const double* W, long long W_bs,   /* [U,Ds] */
                        const double* b, long long b_bs,   /* [U]    */
                        const double* m /*[R,Ds]*/, const double* s /*[R,Ds,Ds]*/,
                        double* M /*[R,U]*/, double* S /*[R,U,U]*/, double* V /*[R,Ds,U]*/,
                        pilco_stream_t stream);

int pilco_exp_reward(int Ds, int R, const double* W /*[Ds,Ds]*/, const double* t /*[Ds]*/,
                     const double* m /*[R,Ds]*/, const double* s /*[R,Ds,Ds]*/,
                     double* muR /*[R]*/, double* sR /*[R] or NULL*/, int* info,
                     pilco_stream_t stream);

/* Safe-PILCO risk rewards (safe_pilco_extension/rewards_safe.py:13-58: RiskOfCollision.compute_reward,
 * SingleConstraint.compute_reward): probability that the constrained state dimensions lie inside a box,
 * each dimension an independent univariate normal with loc m[d] and scale sfac*s[d,d] (as the reference
 * writes it).  prm (device, doubles) = [nd, inside, sfac, (dim_k, low_k, high_k) x nd]; a missing bound is
 * +-inf; inside = 0 returns the complement.  Optional d risk/d m [R,Ds] and d risk/d diag(s) [R,Ds]. */
int pilco_box_risk(int Ds, int R, const double* prm, const double* m /*[R,Ds]*/, const double* s /*[R,Ds,Ds]*/,
                   double* risk /*[R]*/, double* drisk_dm /*[R,Ds] or NULL*/, double* drisk_dv /*[R,Ds] or NULL*/,
                   pilco_stream_t stream);

/* ---- H-step rollout ---------------------------------------------------------------------------
 * Replaces PILCO.predict / PILCO.propagate (pilco/models/pilco.py:118-153; pred.m:29-39,
 * propagate.m:33-85): policy moments -> joint state/action Gaussian -> dynamics moment match ->
 * next state; the expected reward is accumulated at the pre-step state (pilco.py:130-134).
 */
#define PILCO_POLICY_LINEAR 0
#define PILCO_POLICY_RBF    1
#define PILCO_REWARD_EXP    0
#define PILCO_REWARD_LINEAR 1
#define PILCO_REWARD_BOX    2   /* pilco_box_risk; W = its prm block, t unused */
/* accumulation channel of a reward term (safe_pilco_extension/safe_pilco.py:29-50, SafePILCO.predict):
 *   ADD : reward_add  += coef * value(x_t)                       (PILCO.predict, pilco.py:130-134)
 *   MULT: reward_mult *= 1 - sum_k coef_k * value_k(x_t)          (the terms of this channel form the risk)
 * and the rollout returns  reward = reward_add + mult_mu * (1 - reward_mult). */
#define PILCO_CHANNEL_ADD   0
#define PILCO_CHANNEL_MULT  1

typedef struct pilco_policy {
    int kind;                   /* PILCO_POLICY_* */
    int Ds, U;
    int squash;                 /* 1: squash_sin with max_action */
    const double* max_action;   /* [U] */
    /* linear (controllers.py:39-63) */
    const double* W; long long W_bs;   /* [U,Ds] */
    const double* b; long long b_bs;   /* [U]    */
    /* RBF (controllers.py:80-129): deterministic GP over bf centres; beta from pilco_gp_factorize */
    pilco_gp_model rbf;
} pilco_policy;

typedef struct pilco_reward_term {
    int kind;                   /* PILCO_REWARD_* */
    int channel;                /* PILCO_CHANNEL_* */
    double coef;                /* CombinedRewards weight (rewards.py:64-81) */
    const double* W;            /* exp: [Ds,Ds]; linear: [Ds]; box: prm block */
    const double* t;            /* exp: [Ds] target; linear: unused */
} pilco_reward_term;

typedef struct pilco_rollout {
    int R, H;
    pilco_gp_model dyn;         /* D = Ds+U, E = Ds */
    pilco_policy   pol;
    int n_rewards;
    pilco_reward_term rewards[8];
    const double* m0; long long m0_bs;   /* [Ds]    initial state mean  */
    const double* S0; long long S0_bs;   /* [Ds,Ds] initial state cov   */
    /* outputs */
    double* traj_m;             /* [R,H+1,Ds]    state means, t=0..H   */
    double* traj_S;             /* [R,H+1,Ds,Ds] state covariances      */
    double* reward;             /* [R] sum_{t<H} E[r(x_t)]  (+ mult_mu (1 - prod_t (1 - risk_t)))  */
    double* step_reward;        /* [R,H] or NULL                        */
    int* info;                  /* [R]                                   */
    void* ws; size_t ws_bytes;
    double mult_mu;             /* SafePILCO.mu (safe_pilco.py:26,49); ignored without MULT terms */
    double* step_risk;          /* [R,H] per-step risk of the MULT channel, or NULL */
    /* Tape of the dynamics moment match (pilco_rollout_tape_bytes, 16-byte aligned) or NULL.  With a tape the forward
     * cascade runs the TAPED tile pass (pilco_mm_forward_taped) at every step and pilco_rollout_backward consumes
     * the tape instead of recomputing any N x N exponential: forward+backward cost ~1.9 forward tile passes instead
     * of ~5.  Without it pilco_rollout_backward recomputes (memory-lean path, same results). */
    void* tape; size_t tape_bytes;
} pilco_rollout;

size_t pilco_rollout_workspace_bytes(const pilco_rollout* ro);
size_t pilco_rollout_tape_bytes(const pilco_rollout* ro);   /* 0: shape not supported by the taped pass (n > 1024 centres for D <= 12, > 704 beyond) */
int    pilco_rollout_forward(const pilco_rollout* ro, pilco_stream_t stream);

/* Reverse sweep: gradient of ro->reward[r] (= sum_t E[r(x_t)], the negative of PILCO.training_loss,
 * pilco/models/pilco.py:47-50) with respect to the policy parameters.  Must follow pilco_rollout_forward
 * with the same `ro` (the per-step joint Gaussians it saved in ro->ws are re-used).
 * Linear policy: gW [R,U,Ds], gb [R,U].  RBF policy: gXc [R,bf,Ds] centres, gYc [R,bf,U] targets,
 * gell [R,U,Ds] lengthscales (constrained), pol_L = Cholesky factors left by pilco_gp_factorize. */
typedef struct pilco_rollout_grad {
    double* gW; double* gb;
    double* gXc; double* gYc; double* gell;
    const double* pol_L;
    double* gm0; double* gS0;       /* optional: gradient w.r.t. the initial state moments [R,Ds],[R,Ds,Ds] */
    void* ws; size_t ws_bytes;
} pilco_rollout_grad;

size_t pilco_rollout_bwd_workspace_bytes(const pilco_rollout* ro);
int    pilco_rollout_backward(const pilco_rollout* ro, const pilco_rollout_grad* g, pilco_stream_t stream);

/* ---- diagnostics ------------------------------------------------------------------------------
 * fp64 pipe microbenchmark used for the roofline denominators (DESIGN.md "Roofline"): which = 0 DFMA,
 * 1 DMMA m8n8k4, 2 both interleaved, 3 table exp, 4 libdevice exp; 8 ops/thread/iteration (16 DMMA for
 * which=1,2 counted as 8 pairs).  Synchronises (it times itself with CUDA events) -- never call it in a
 * captured region. */
/* pilco_mm_forward with CUDA events around its three launches: ms_out[0..2] = setup, tile, finish.
 * Synchronises. */
int pilco_mm_forward_profile(const pilco_gp_model* gp, int R, const double* m, const double* s,
                             double* M, double* S, double* V, int* info,
                             void* ws, size_t ws_bytes, float* ms_out, pilco_stream_t stream);
int pilco_mm_forward_taped_profile(const pilco_gp_model* gp, int R, const double* m, const double* s,
                                   double* M, double* S, double* V, int* info,
                                   void* ws, size_t ws_bytes, void* tape, size_t tape_bytes,
                                   float* ms_out, pilco_stream_t stream);
int pilco_microbench_fp64(int which, int iters, int blocks, double* sink_dev, float* ms_out, pilco_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* PILCO_B200_H */
