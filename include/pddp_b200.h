/* pddp_b200 -- C ABI of the B200-native iLQR / PDDP iteration hot path.
 *
 * The reference (anassinator/pddp) is pure Python: its "FFI" for this path is the set of
 * module-level functions in pddp/controllers/ilqr.py that the controller calls once per
 * iteration.  Each entry point below replaces one of them for a BATCH of independent problems;
 * the citation after each declaration is the reference interface it stands in for.
 *
 * Conventions
 *   - plain C: device pointers + sizes + a cudaStream_t passed as void*.  No allocation inside,
 *     the caller owns every buffer; all work is enqueued on `stream` and nothing synchronises.
 *   - return value: 0 on success, a negative PDDP_E_* code for bad arguments / unsupported
 *     configurations, a positive value = cudaError_t of a failed launch.
 *     pddp_last_error() returns a thread-local message.  Per-problem numerical outcomes
 *     (not-positive-definite, NaN) are reported in int32 status buffers, never as errors.
 *   - dtype: PDDP_F32 / PDDP_F64 element type of every floating-point buffer in the call.
 *   - tensors are [B, Nt, E] (problem b, time t, element e) in one of two layouts:
 *       PDDP_PROBLEM_MAJOR  offset = (b*Nt + t)*E + e      (reference layout + leading B)
 *       PDDP_BATCH_INNER    offset = (t*E + e)*B + b       (SoA over problems)
 *     Matrices are row-major inside E (F_z[r][c] -> e = r*nz + c, K[i][c] -> e = i*nz + c).
 *   - safe to call from one host thread per device.
 */
#ifndef PDDP_B200_H
#define PDDP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PDDP_F32 0
#define PDDP_F64 1

#define PDDP_PROBLEM_MAJOR 0
#define PDDP_BATCH_INNER 1

/* pddp/utils/encoding.py:25-33 (StateEncoding) */
#define PDDP_ENC_FULL_COVARIANCE_MATRIX 0
#define PDDP_ENC_UPPER_TRIANGULAR_CHOLESKY 1
#define PDDP_ENC_VARIANCE_ONLY 2
#define PDDP_ENC_STANDARD_DEVIATION_ONLY 3
#define PDDP_ENC_IGNORE_UNCERTAINTY 4

/* state geometry (which dims are angles): pddp/examples/{pendulum,cartpole,double_cartpole}/model.py */
#define PDDP_GEO_PENDULUM 0        /* D=2, angles {0}      */
#define PDDP_GEO_CARTPOLE 1        /* D=4, angles {2}      */
#define PDDP_GEO_DOUBLE_CARTPOLE 2 /* D=6, angles {2,4}    */
#define PDDP_GEO_RENDEZVOUS 3      /* D=8, no angles, action_size 4 (pddp/examples/rendezvous/model.py; known and BNN dynamics) */

/* pddp/controllers/ilqr.py:35-64 (iLQRState) */
#define PDDP_STATE_UNDEFINED 0
#define PDDP_STATE_ACCEPTED 1
#define PDDP_STATE_REJECTED 2
#define PDDP_STATE_NOT_PD 3
#define PDDP_STATE_MAX_REG 4
#define PDDP_STATE_CONVERGED 5

/* backward / rollout status bits */
#define PDDP_OK 0
#define PDDP_STATUS_NOT_PD 1   /* reference: RuntimeError in backward (ilqr.py:639-640,653-655) */
#define PDDP_STATUS_NAN 2      /* reference: exception out of _control_law / Cholesky failure   */

#define PDDP_E_BADARG (-1)
#define PDDP_E_UNSUPPORTED (-2)

#define PDDP_MAX_DA 8
#define PDDP_MAX_NU 4

/* Problem shape shared by all calls. */
typedef struct pddp_shape {
    int32_t dtype;   /* PDDP_F32 | PDDP_F64 */
    int32_t layout;  /* PDDP_PROBLEM_MAJOR | PDDP_BATCH_INNER */
    int32_t geo;     /* PDDP_GEO_* */
    int32_t enc;     /* PDDP_ENC_* */
    int32_t B;       /* independent problems */
    int32_t N;       /* horizon */
    int32_t nz;      /* encoded state size (must equal the encoding's size for geo's D) */
    int32_t nu;      /* action size of the geometry: 1 for the three pendulum-family geometries, 4 for rendezvous */
} pddp_shape;

/* Constants of a QRCost on the angle-augmented state (host memory, doubles, row-major DAxDA).
 * Replaces: pddp/costs/quadratic.py:39-58 + pddp/examples/<problem>/cost.py constructor. */
typedef struct pddp_cost {
    double Q[PDDP_MAX_DA * PDDP_MAX_DA];
    double Q_term[PDDP_MAX_DA * PDDP_MAX_DA];
    double R[PDDP_MAX_NU * PDDP_MAX_NU];   /* row-major nu x nu (stride nu) */
    double x_goal[PDDP_MAX_DA];
    double u_goal[PDDP_MAX_NU];
} pddp_cost;

/* Known-dynamics constants (host memory). p[] = pendulum: dt,m,l,mu,g ; cartpole: dt,mc,mp,l,mu,g ;
 * double cartpole: dt,mc,mp1,mp2,l1,l2,mu,g ; rendezvous: dt,m,alpha.
 * Replaces: pddp/examples/<problem>/model.py constructor Parameters. */
typedef struct pddp_known_dynamics {
    double p[8];
} pddp_known_dynamics;

/* Input particles of step i (pddp/models/bnn/modules.py:320-358):
 *   INFER    infer_noise_variables=True (default): step 0 uses m + eps_in[0] U, step i>0 re-uses the output
 *            particles of step i-1 (eps = (X - m) U^-1 held constant in the derivatives)
 *   RESAMPLE infer_noise_variables=False: X = m + eps_in[i] U(z_i) at every step
 *   MEAN     sample_input_distribution=False: every particle starts at the mean (the covariance is ignored) */
#define PDDP_BNN_INPUT_INFER 0
#define PDDP_BNN_INPUT_RESAMPLE 1
#define PDDP_BNN_INPUT_MEAN 2

/* Eval-mode BNN dynamics (device pointers, element type = shape.dtype).
 * Replaces the state read by pddp/models/bnn/modules.py:200-264,287-386:
 * Linear weights (torch [out,in] row-major), persistent dropout masks [P,H] (SURVEY quirk 8-10),
 * eps_in[0] [P,D], normalisation buffers (NULL = 0 / 1 defaults). Two hidden layers. */
typedef struct pddp_bnn {
    int32_t P;            /* particles */
    int32_t H0, H1;       /* hidden widths */
    const void* W0; const void* b0;   /* [H0, DA+nu], [H0] */
    const void* W1; const void* b1;   /* [H1, H0], [H1]    */
    const void* W2; const void* b2;   /* [2D, H1], [2D]  (only the first D rows are used) */
    const void* mask0;    /* [P, H0] */
    const void* mask1;    /* [P, H1] */
    const void* eps0;     /* [P, D]  */
    const void* X_mean; const void* X_std_inv;  /* [DA+nu] or NULL */
    const void* dX_mean; const void* dX_std;    /* [D] or NULL */
    int32_t input_mode;   /* PDDP_BNN_INPUT_* : how the input particles of step i are formed */
    const void* eps_in;   /* [N, P, D] standardised noise of every step (PDDP_BNN_INPUT_RESAMPLE only;
                             the reference draws eps_in[i] lazily, modules.py:321-329 -- here it is data) */
    const void* eps_out;  /* [N, P, D] or NULL.  Non-NULL = use_predicted_std=True (modules.py:242-262):
                             dX_std * exp(log_std head) * eps_out[i] is added to every particle; runs the
                             CUDA-core MLP kernel (the tcgen05 kernel evaluates the mean head only) */
    int32_t independent_noise;  /* with eps_out: exp(log_std) is treated as a constant in the derivatives */
} pddp_bnn;

const char* pddp_version(void);
const char* pddp_last_error(void);

/* ---- linearise: nominal rollout + all derivatives ------------------------------------------
 * Replaces pddp.controllers.ilqr.forward (ilqr.py:393-486) and, inside it,
 * batch_eval_cost / batch_eval_dynamics (pddp/utils/evaluation.py:134-288).
 *   in : z0[B,nz]  U[B,N,nu]  u_min/u_max[nu] device pointers or NULL (no clamping)
 *        active[B] int32 or NULL: problems with active==0 are skipped (their outputs keep
 *        the previous linearisation -- the reference's retry loop, ilqr.py:213-233)
 *   out: Z[B,N+1,nz] F_z[B,N,nz*nz] F_u[B,N,nz*nu] L[B,N+1,1] L_z[B,N+1,nz] L_u[B,N,nu]
 *        L_zz[B,N+1,nz*nz] L_uz[B,N,nu*nz] L_uu[B,N,nu*nu]  J_opt[B] = sum_t L
 *        status[B] |= PDDP_STATUS_NAN when a non-finite value appears                          */
int pddp_linearize_known(const pddp_shape* shape, const pddp_known_dynamics* dyn,
                         const pddp_cost* cost, const void* z0, const void* U, const void* u_min,
                         const void* u_max, const int32_t* active, void* Z, void* F_z, void* F_u,
                         void* L, void* L_z, void* L_u, void* L_zz, void* L_uz, void* L_uu,
                         void* J_opt, int32_t* status, void* stream);

/* ---- backward Riccati pass ------------------------------------------------------------------
 * Replaces pddp.controllers.ilqr.backward + Q (ilqr.py:489-674, default V_zz_reg=False branch)
 * and, with bounds, pddp.utils.constraint.boxqp (constraint.py:150-266).  This call only needs the
 * derivative tensors: shape.geo / shape.enc are ignored and any nz >= 1, 1 <= nu <= PDDP_MAX_NU is
 * accepted (nu > 1: eigen-clipping by Jacobi rotations and the n-dimensional projected-Newton box QP;
 * u_min / u_max are [nu] vectors).
 *   in : the derivative tensors above, mu[B] (per-problem regularisation, float64), U,
 *        u_min/u_max or NULL
 *   out: k[B,N,nu]  K[B,N,nu*nz]  status[B] = PDDP_STATUS_NOT_PD where the reference would raise */
int pddp_backward(const pddp_shape* shape, const void* F_z, const void* F_u, const void* L_z,
                  const void* L_u, const void* L_zz, const void* L_uz, const void* L_uu,
                  const double* mu, const void* U, const void* u_min, const void* u_max,
                  const int32_t* active, void* k, void* K, int32_t* status, void* stream);

/* ---- forward rollout with parallel line search + trajectory cost ---------------------------
 * Replaces pddp.controllers.ilqr._control_law + _trajectory_cost + the argmin in _step
 * (ilqr.py:677-723, 764-791, 161-164) for known dynamics.
 *   in : Z,U nominal, k,K gains, alphas[A] (device), bounds or NULL, bw_status[B] (problems whose
 *        backward pass failed are skipped)
 *   out: J_all[B,A] cost of every alpha, amin[B], J_new[B] = min, Z_new[B,N+1,nz], U_new[B,N,nu]
 *        (the winning alpha's trajectory)                                                       */
int pddp_rollout_known(const pddp_shape* shape, const pddp_known_dynamics* dyn,
                       const pddp_cost* cost, const void* Z, const void* U, const void* k,
                       const void* K, const void* alphas, int32_t A, const void* u_min,
                       const void* u_max, const int32_t* active, const int32_t* bw_status,
                       void* J_all, int32_t* amin, void* J_new, void* Z_new, void* U_new,
                       void* stream);

/* ---- per-problem accept / reject + regularisation schedule ---------------------------------
 * Replaces the tail of iLQRController._step and _reset/_decrease/_increase_reg
 * (ilqr.py:166-181, 364-390), vectorised over problems, plus the copy of the accepted candidate
 * into the nominal trajectory (self._Z_nominal/_U_nominal, ilqr.py:167-168).
 *   inout: mu[B], delta[B] (doubles always), J_opt[B], state[B], iters_left[B], active[B], Z, U
 *   in   : J_new[B], bw_status[B], Z_new, U_new, tol, max_reg
 *          active[b]: 0 = finished, 1 = needs a fresh linearisation, 2 = retry backward+rollout
 *          on the existing linearisation with the increased mu (ilqr.py:213-233)
 *   out  : accepted[B] (1 where the candidate was taken), n_active[1] int32 incremented by the
 *          number of problems that still need passes (may be NULL)
 *   K, K_nominal (both or neither, [B,N,nu*nz]): the gains of THIS backward pass are copied into
 *          K_nominal only where the candidate was accepted -- the reference stores self._K on an accepted
 *          step only (ilqr.py:166-171), so after a fit that ends in MAX_REG the feedback law still uses
 *          the gains of the last accepted step, not those of the rejected high-mu retries.           */
int pddp_accept_update(const pddp_shape* shape, const void* J_new, const int32_t* bw_status,
                       const void* Z_new, const void* U_new, double tol, double max_reg, double* mu,
                       double* delta, void* J_opt, int32_t* state, int32_t* iters_left,
                       int32_t* active, void* Z, void* U, int32_t* accepted, int32_t* n_active,
                       const void* K, void* K_nominal, void* stream);

/* ---- BNN dynamics ----------------------------------------------------------------------------
 * pddp_linearize_bnn replaces ilqr.forward with a factory-built BNNDynamicsModel
 * (pddp/models/bnn/modules.py:287-386 + 200-264, eval mode; the infer_noise_variables /
 * sample_input_distribution options are pddp_bnn.input_mode, use_predicted_std is pddp_bnn.eps_out); pddp_rollout_bnn replaces
 * _control_law + _trajectory_cost for the same model.  `workspace` is a device scratch buffer of
 * at least pddp_bnn_workspace_bytes(...) bytes.  Every geometry has BNN kernels; shape.nu must be its
 * action size, and U / u_min / u_max / k / K / F_u carry all nu components.  The rendezvous cost is the
 * plain QR cost on the state (no angle augmentation), as in the known-dynamics path.          */
int64_t pddp_bnn_workspace_bytes(const pddp_shape* shape, const pddp_bnn* bnn, int32_t A);

int pddp_linearize_bnn(const pddp_shape* shape, const pddp_bnn* bnn, const pddp_cost* cost,
                       const void* z0, const void* U, const void* u_min, const void* u_max,
                       const int32_t* active, void* Z, void* F_z, void* F_u, void* L, void* L_z,
                       void* L_u, void* L_zz, void* L_uz, void* L_uu, void* J_opt, int32_t* status,
                       void* workspace, int64_t workspace_bytes, void* stream);

int pddp_rollout_bnn(const pddp_shape* shape, const pddp_bnn* bnn, const pddp_cost* cost,
                     const void* Z, const void* U, const void* k, const void* K, const void* alphas,
                     int32_t A, const void* u_min, const void* u_max, const int32_t* active,
                     const int32_t* bw_status, void* J_all, int32_t* amin, void* J_new, void* Z_new,
                     void* U_new, int32_t* status, void* workspace, int64_t workspace_bytes,
                     void* stream);

/* Cost value / gradient / Hessian of a batch of encoded states (used by the BNN linearise pass,
 * exported for testing).  Replaces batch_eval_cost (pddp/utils/evaluation.py:134-239).
 *   in : Z[B,N+1,nz], U[B,N,nu] (already clamped);  out: L, L_z, L_u, L_zz, L_uz, L_uu, J_opt    */
int pddp_cost_derivatives(const pddp_shape* shape, const pddp_cost* cost, const void* Z,
                          const void* U, const int32_t* active, void* L, void* L_z, void* L_u,
                          void* L_zz, void* L_uz, void* L_uu, void* J_opt, void* stream);

/* ---- ground-truth simulator step (closed-loop MPC / trials) ----------------------------------------
 * Replaces the step() of the example environments (pddp/examples/<problem>/env.py: x' = model(x, u, 0,
 * IGNORE_UNCERTAINTY)) behind GymEnv.apply (pddp/envs/gym_env.py:63-73) for B environment instances at
 * once, so that pddp.controllers.pddp._apply_controller (pddp.py:209-247) never leaves the device.
 *   in : x[B, D] states, u[B, nu] actions (shape.geo, shape.dtype, shape.B are read; the rest is ignored)
 *   out: x_next[B, D]  (may alias x)                                                                  */
int pddp_env_step_known(const pddp_shape* shape, const pddp_known_dynamics* dyn, const void* x, const void* u,
                        void* x_next, void* stream);

/* ---- BNN training on the device (SURVEY 8f rank 4) -------------------------------------------------
 * Replaces the optimisation loop of ParticlesBNNDynamicsModel.fit (pddp/models/bnn/modules.py:174-198):
 * n_iter steps of torch.optim.Adam(amsgrad=True) on
 *     -gaussian_log_likelihood(dX, mean, exp(log_std)).mean() + reg_scale * model.regularization() / n_data
 * (pddp/models/bnn/losses.py:20-38; regulariser modules.py:434-447, 517-530, 749-766: drop_0 weighs fc_1,
 * drop_1 weighs fc_out, with keep-probability 1 - rate: the learned logit_p never reaches it, see
 * csrc/bnn_train.cu), the network evaluated in training mode with
 * a fresh dropout mask per (row, unit) and step (modules.py:462-483, 550-583, resample=True).
 *   params  flat [W0[H0,K0] | b0[H0] | W1[H1,H0] | b1[H1] | W2[2D,H1] | b2[2D] | logit_p0 | logit_p1]
 *           (torch layouts; logit_p only for dropout == 0), updated in place
 *   X [n_data,K0] augmented state + action (un-normalised), dX [n_data,D] targets; X_mean / X_std_inv [K0],
 *   dX_mean / dX_std [D] normalisation buffers or NULL pairs (0 / 1)
 *   batch_idx [n_iter,batch] int32 rows of the step's mini-batch, -1 = empty slot (partial last batch)
 *   noise   [n_iter,batch,H0+H1] uniforms for the masks, or NULL: counter-based generator from cfg.seed
 *   grads   gradient of the LAST step (same layout as params), loss [n_iter] the loss of every step        */
typedef struct pddp_bnn_train_config {
    int32_t dtype;                 /* PDDP_F32 | PDDP_F64 */
    int32_t K0, H0, H1, D;         /* input width DA+nu, hidden widths, state size (output width 2D) */
    int32_t n_data, batch, n_iter;
    int32_t dropout;               /* 0 = CDropout (concrete, learns logit_p), 1 = BDropout (Bernoulli(1-rate)) */
    double lr, beta1, beta2, eps;  /* Adam */
    double reg_scale, temperature;
    double reg0, reg1;             /* BDropout.reg of drop_0 / drop_1 */
    double rate0, rate1;           /* BDropout.rate of drop_0 / drop_1 (both kinds: the regulariser uses 1 - rate) */
    uint64_t seed;
} pddp_bnn_train_config;

int64_t pddp_bnn_train_workspace_bytes(const pddp_bnn_train_config* cfg);

int pddp_bnn_train(const pddp_bnn_train_config* cfg, const void* X, const void* dX, const void* X_mean,
                   const void* X_std_inv, const void* dX_mean, const void* dX_std, const int32_t* batch_idx,
                   const void* noise, void* params, void* grads, void* loss, void* workspace,
                   int64_t workspace_bytes, void* stream);

/* ---- instrumentation (bench.py) -----------------------------------------------------------------
 * pddp_profile_enable(1) makes the BNN path bracket its kernels with CUDA events on the launch
 * stream; pddp_profile_read synchronises and returns total milliseconds / launch counts for
 * kind 0 = MLP (linearise), 1 = MLP (rollout), 2 = moment matching (linearise), 3 = rollout step,
 * 4 = backward pass, 5 = cost derivatives, 6 = linearise (known dynamics), 7 = rollout (known dynamics),
 * 8 = accept / copy; `ms` and `count` must hold PDDP_PROFILE_KINDS entries.
 * pddp_launch_count() = kernels launched by this library since load.                          */
#define PDDP_PROFILE_KINDS 9
void pddp_profile_enable(int on);
int pddp_profile_read(double* ms, int64_t* count);
int64_t pddp_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* PDDP_B200_H */
