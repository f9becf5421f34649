/* mobocmf_b200 — C ABI of the B200-native MFDGP hot path (sm_100a).
 *
 * The reference (fernandezdaniel/MOBOCMF) has no FFI: its boundary is the Python class API (SURVEY.md §8b).  These
 * entry points are what a binding for that path would call; each cites the reference code it replaces.  All
 * pointers are DEVICE pointers to fp64 unless stated; sizes are explicit; `stream` is a cudaStream_t passed as
 * void*.  Every function returns 0 on success, -1 on a CUDA launch error, -2 on an unsupported shape
 * (M > 256, d > 8).  No function synchronises or allocates device memory; scratch is caller-provided.  State kept by
 * the library: launch counters / the optional profile log, and the side stream + events of the fused step, which live
 * in a caller-owned step context (mobo_step_ctx_create) or, for callers that pass none, in one lazily created
 * per-device default.
 *
 * Conventions
 *   kind 0  layer-0 covariance  a * RBF_ARD(x)                       (mobocmf/layers/mfdgp_hidden_layer.py:43-47)
 *           theta = [a, l_0 .. l_{d-1}]
 *   kind 1  layer>=1 covariance k_x1 * (k_lin + k_f) + k_x2 on [x, f] (mobocmf/layers/mfdgp_hidden_layer.py:70-88,115)
 *           theta = [a1, v_lin, a_f, l_f, a2, l1_0 .. l1_{d-1}, l2_0 .. l2_{d-1}]
 *   theta holds CONSTRAINED values (softplus already applied); d = number of x columns (without f).
 *   MP = M rounded up to a multiple of 32.  An "operator buffer" is mobo_ops_doubles(M) doubles laid out as
 *   [L | W | WT | H | HT | P | LQ] (seven MP x MP row-major blocks), [WF | HTF | HF | WTF] (W, HT, H, WT again in the
 *   DMMA A-fragment order the row kernels stream them in), beta[MP], alpha[MP], scal[16], rowstat[4 MP], flags[128]
 *   (scal[0] = KL, scal[5] = Cholesky status: 0 ok, 1 not positive definite after the three psd_safe_cholesky
 *   retries with 1e-8, 1e-7, 1e-6 more on the diagonal, scal[7] = retries used).
 *   The GRADIENT of an operator buffer uses the same layout and, by convention, carries only
 *   block W: A2 = sum_r dvar_r t_r t_r^T (t = W k, whitened), block H: the same sum over clamped rows,
 *   alpha: b = sum_r dmu_r t_r,
 *   scal[0]: d loss / d KL, scal[6]: number of clamped rows behind block H.
 */
#ifndef MOBOCMF_B200_H
#define MOBOCMF_B200_H
#include <stddef.h>
#ifdef __cplusplus
extern "C" {
#endif

/* library / build identification: 103 (sm_100a; 100 + ABI revision; 2: mobo_step_desc.ctx, step contexts;
 * 3: the multi-layer operator-chain entry points and the stand-alone K(Z, Z) entry point removed, more scratch for
 * mobo_layer_rows_bwd) */
int mobo_abi_version(void);

/* Launch accounting: number of kernels this library has launched in this process; optional per-launch CUDA-event
 * timing (enable, run, then collect: NUL-separated kernel names into `names`, milliseconds into `ms`; returns the
 * number of records written and clears the log).  Used by bench.py for `gpu_launches` and the roofline kernel. */
long long mobo_launch_count(void);
void mobo_profile_enable(int on);
int mobo_profile_collect(char* names, size_t names_bytes, float* ms, int max_records);

int mobo_padded_m(int M);
size_t mobo_ops_doubles(int M);
/* doubles needed for each of Tsave / Usave of mobo_layer_rows_fwd for R rows */
size_t mobo_rows_save_doubles(int M, long long R);
/* scratch doubles for mobo_layer_rows_bwd / mobo_layer_precompute_bwd */
size_t mobo_rows_bwd_work_doubles(int M, long long R);
size_t mobo_precompute_bwd_work_doubles(int M);

/* Per-step operators of one sparse-GP layer.
 * Replaces: UnwhitenedVariationalStrategy.forward's K_zz + jitter, Cholesky and solves, and kl_mvn_mvn
 * [upstream gpytorch], reached from mobocmf/layers/mfdgp_hidden_layer.py:286 and
 * mobocmf/mlls/variational_elbo_mf.py:40; jitter = CovarianceMatrixMF.add_jitter (layers/...py:17-20).
 * Zx: M x d; zf: M (kind 1: previous layer's variational mean, layers/...py:556-557) or NULL;
 * m: M variational mean; Lq: M x M chol_variational_covar (tril applied inside). */
int mobo_layer_precompute(int kind, int d, int M, const double* Zx, const double* zf, const double* theta,
                          const double* m, const double* Lq, double jitter, double* ops, void* stream);

/* Backward of mobo_layer_precompute.  gops: gradient buffer (convention above).  work:
 * mobo_precompute_bwd_work_doubles(M).  Outputs: dtheta[theta size], dzf[M] (kind 1), dm[M], dLq[M x M]. */
int mobo_layer_precompute_bwd(int kind, int d, int M, const double* Zx, const double* zf, const double* theta,
                              const double* m, const double* Lq, const double* ops, const double* gops,
                              double* work, double* dtheta, double* dzf, double* dm, double* dLq, void* stream);

/* Fused row pass of one layer: K(Z_l, X) in shared memory -> mean / variance of q(f) for R rows, with the
 * reparameterised propagation of the previous layer's sample fused in.
 * Replaces: MFDGPHiddenLayer.__call__ / forward (mobocmf/layers/mfdgp_hidden_layer.py:232-286) and
 * UnwhitenedVariationalStrategy.forward's mean/variance [upstream].
 * x: n x d, row r reads x[r / xrep].  kind 1: f_r = f_direct[r] if f_direct else
 * mu_prev[r / prep] + sqrt(max(var_prev[r / prep], 1e-10)) * eps[r % eps_mod].
 * training != 0 selects clamp(k_xx - q, 0).  craw (optional): k_xx - q before the clamp; clamp_count (optional,
 * device unsigned): incremented per clamped row.  Tsave/Usave (optional, both or none): t = W k and u = H^T t saved for the
 * backward, mobo_rows_save_doubles(M, R) doubles each. */
int mobo_layer_rows_fwd(int kind, int d, int M, const double* Zx, const double* zf, const double* theta,
                        const double* ops, const double* x, int xrep, const double* mu_prev, const double* var_prev,
                        int prep, const double* eps, long long eps_mod, const double* f_direct, long long R,
                        int training, double* mu, double* var, double* craw, unsigned int* clamp_count,
                        double* Tsave, double* Usave, void* stream);

/* Backward of mobo_layer_rows_fwd given dmu[R], dvar[R].
 * Outputs: df[R] (kind 1; d loss / d f_r), dxrow[R x d] (optional, d loss / d x per row), dtheta, dzf[M]
 * (want_param_grads), and the A2 / Ac / dalpha entries of the operator-gradient buffer gops (other entries of
 * gops are left untouched).  work: mobo_rows_bwd_work_doubles(M, R). */
int mobo_layer_rows_bwd(int kind, int d, int M, const double* Zx, const double* zf, const double* theta,
                        const double* ops, const double* x, int xrep, const double* mu_prev, const double* var_prev,
                        int prep, const double* eps, long long eps_mod, const double* f_direct, long long R,
                        int training, const double* dmu, const double* dvar, const double* craw,
                        const unsigned int* clamp_count, const double* Tsave,
                        const double* Usave, int want_param_grads, double* df, double* dxrow, double* dtheta,
                        double* dzf, double* gops, double* work, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Fused ELBO step: the body of BlackBoxMFDGPFitter._update_model up to the gradients
 * (mobocmf/util/blackbox_mfdgp_fitter.py:161-168: model(x), elbo(output, y.T, fid), loss = -elbo, loss.backward())
 * as ONE enqueue of kernels without host synchronisation (CUDA-graph capturable):
 * constraint transforms (softplus / Interval sigmoid, mobocmf/models/mfdgp.py:116), operator chain of every layer,
 * the L fused row passes (MFDGP.forward, mobocmf/models/mfdgp.py:174-196), the ELBO
 * (VariationalELBOMF.forward, mobocmf/mlls/variational_elbo_mf.py:24-51), the complete backward and the assembly of
 * d loss / d RAW parameter.  Preconditions (the host mirror checks them and otherwise uses the composable entry
 * points above): every layer shares the inducing inputs Zx (quirk Q4, so Z_l = [Zx, m_{l-1}]), training mode.
 * S > 1 (not in the reference, SURVEY.md F4): layer 0 on B rows, layers >= 1 on B*S rows (row b*S+s), data terms
 * averaged over s.  All pointers are device pointers.
 * ------------------------------------------------------------------------------------------------------------ */
#define MOBO_MAX_LAYERS 8
#define MOBO_MAX_THETA 21            /* 5 + 2 * 8 */

typedef struct mobo_layer_desc {
  const double* Zx;                            /* M x d shared inducing inputs                                  */
  const double* raw_theta[MOBO_MAX_THETA];     /* address of each RAW kernel hyper-parameter, in theta order     */
  double* g_raw_theta[MOBO_MAX_THETA];         /* where d loss / d raw goes; NULL = frozen                       */
  const double* m;                             /* variational_mean [M]                                           */
  const double* Lq;                            /* chol_variational_covar [M x M] (tril applied inside)           */
  double* g_m;                                 /* NULL = frozen                                                  */
  double* g_Lq;                                /* NULL = frozen; receives the lower triangle, zeros above        */
  const double* raw_noise;                     /* likelihood raw_noise [1]                                       */
  double* g_raw_noise;                         /* NULL = frozen                                                  */
  double noise_lower, noise_upper;             /* Interval bounds (mobocmf/models/mfdgp.py:116)                  */
  const double* eps;                           /* layer >= 1: B*S standard normals (layers/...py:274); layer 0: NULL */
} mobo_layer_desc;

typedef struct mobo_step_desc {
  int L, d, M, S;
  long long B, num_data;
  double jitter;
  const double* x;                             /* B x d                                                          */
  const double* y;                             /* B                                                              */
  const double* fid;                           /* B, fidelity index stored as double (as the reference does)     */
  mobo_layer_desc layer[MOBO_MAX_LAYERS];
  double* out;                                 /* 8 doubles: [0] loss = -ELBO, [1] KL*B/N, [2] data term, [3] status:
                                                  0 ok, l+1 = Cholesky of layer l failed after psd_safe_cholesky's
                                                  three jitter retries (NotPSDError upstream); [4] first non-zero
                                                  status since the caller last zeroed it (sticky); [5] sticky "loss not
                                                  finite" (NanError upstream); [6] 1 when THIS step failed either way
                                                  (pass &out[6] to mobo_adam as skip_flag); [7] retries used (0..3)  */
  double* workspace;                           /* mobo_elbo_step_workspace_doubles(...) doubles                  */
  int accumulate;                              /* 0: gradients are overwritten, 1: added to                      */
  void* ctx;                                   /* mobo_step_ctx_create() handle (side stream + events of this caller) or
                                                  NULL: the per-device default context                              */
} mobo_step_desc;

size_t mobo_elbo_step_workspace_doubles(int L, int d, int M, int S, long long B);
/* Step context: the side stream (non-blocking, on the current device) and the fork / join events with which
 * mobo_elbo_step runs each layer's operator-chain backward behind the row kernels.  One per concurrently stepping
 * caller (models trained on different streams must not share one: their side work would serialise); destroy it after
 * the last step that used it has completed.  Returns NULL on a CUDA error. */
void* mobo_step_ctx_create(void);
void mobo_step_ctx_destroy(void* ctx);
/* Makes `stream` wait until layer `layer`'s operator-chain backward of the LAST mobo_elbo_step enqueued with this
 * context (accumulate == 0) has completed, i.e. until g_Lq of that layer is final - long before the step ends (the
 * layers are processed high -> low).  For multi-GPU callers: the all-reduce of the large M x M gradient blocks can
 * run behind the remaining row kernels; only the small gradients (m, hyper-parameters, noise) must wait for the end
 * of the step.  Returns -2 for a NULL context / bad layer. */
int mobo_step_ctx_wait_layer(void* ctx, int layer, void* stream);
/* 0 serialises everything on the caller's stream (used by bench.py's per-kernel timing leg); default 1. */
void mobo_step_side_stream(int on);
int mobo_elbo_step(const mobo_step_desc* desc, void* stream);

/* ELBO steps of the K black-box models of a BO iteration at the reference's sizes (M <= 64) in one launch: one CTA
 * runs one model's complete step, the work of mobo_elbo_step (BlackBoxMFDGPFitter._update_model,
 * mobocmf/util/blackbox_mfdgp_fitter.py:156-173, for every model that _train_mfdgp trains).  descs[i] has exactly
 * mobo_elbo_step's meaning (out[8], accumulate, NULL gradient = frozen, g_Lq lower triangle with zeros above), except
 * that desc.ctx is ignored: there is no side stream, and mobo_step_ctx_wait_layer does not apply.  desc.workspace:
 * mobo_elbo_step_small_workspace_doubles(...) doubles (not mobo_elbo_step's size).  Preconditions: those of
 * mobo_elbo_step, and M <= 64.  Returns -2 before any launch when n_models < 1 or any descriptor has M outside
 * [1, 64], d outside [1, 8], L outside [1, 8] or B < 1 (the workspace query returns 0 for those).  Up to 8 models go
 * into one launch of small_step_kernel; more models mean more launches.  Each model's result is independent of the
 * others in the launch (fixed summation orders, no atomics).  CUDA-graph capturable. */
size_t mobo_elbo_step_small_workspace_doubles(int L, int d, int M, int S, long long B);
int mobo_elbo_step_small(const mobo_step_desc* descs, int n_models, void* stream);

/* torch.optim.Adam update (mobocmf/util/blackbox_mfdgp_fitter.py:126,132,259; defaults betas (0.9, 0.999),
 * eps 1e-8, no weight decay) of nt <= 64 tensors in one launch.  step = 1-based step count after increment, or, for
 * CUDA-graph replays, step_dev != NULL: a device-resident count (advance it with mobo_adam_tick before each update;
 * `step` is then ignored).  skip_flag (optional, device): when *skip_flag != 0 nothing is updated - the step that
 * produced the gradients failed (upstream raises NotPSDError / NanError before optimizer.step() is reached). */
typedef struct mobo_adam_tensor { double* p; const double* g; double* exp_avg; double* exp_avg_sq; long long n; } mobo_adam_tensor;
int mobo_adam(int nt, const mobo_adam_tensor* tensors, double lr, double beta1, double beta2, double eps,
              long long step, long long* step_dev, const double* skip_flag, void* stream);
int mobo_adam_tick(long long* step_dev, const double* skip_flag, void* stream);

/* Acquisition chain of ONE MFDGP in eval mode: MFDGP.predict_for_acquisition (mobocmf/models/mfdgp.py:237-262) for n
 * candidates x S fixed normals per layer, up to layer `fidelity`, from precomputed operator buffers (the parameters
 * are constants during optimize_acqf).  theta[l]: CONSTRAINED hyper-parameters; samples[l]: S normals of layer l >= 1
 * (layers/...py:161); zf[l]: m_{l-1}.  Outputs out_mu[n], out_var[n].  scratch: 4 * n * S doubles. */
int mobo_acq_moments(int fidelity, int d, int M, int S, long long n, const double* Zx, const double* const* zf,
                     const double* const* theta, const double* const* ops, const double* const* samples,
                     const double* raw_noise, double noise_lower, double noise_upper, const double* X,
                     double* out_mu, double* out_var, double* scratch, void* stream);
/* Backward of mobo_acq_moments: d / dX of the acquisition chain for optimize_acqf, which differentiates
 * _JES_MFDGP.forward with respect to the candidates (MFDGP.predict_for_acquisition, mobocmf/models/mfdgp.py:237-262;
 * acquisition_functions/JESMOC_MFDGP.py:38-52,142-143).  Same inputs as mobo_acq_moments plus the upstream gradients
 * d_mu[n], d_var[n] (either NULL: zero).  Outputs dX[n x d] and, when d_raw_noise != NULL, d_raw_noise[1]
 * (d / d raw_noise of the likelihood, the one parameter the eval-mode chain does not hold constant); accumulate = 1
 * adds to both instead of overwriting them.  Stateless: it recomputes the forward with exactly mobo_acq_moments'
 * arguments (so its moments are bit-identical to the caller's), saving t and u of every layer in `work`, then runs
 * the row backward of every layer; the result is deterministic (fixed summation orders, no atomics).
 * work: mobo_acq_bwd_work_doubles(...) doubles, 16-byte aligned, laid out as these regions in order, each starting
 * at a multiple of 16 doubles, with R_0 = n, R_l = n S (l >= 1), F = fidelity, B(R) = mobo_rows_save_doubles(M, R):
 *   for l = 0 .. F: mu_l[R_l], var_l[R_l], T_l[B(R_l)], U_l[B(R_l)], dxrow_l[R_l d];
 *   then dmu[R_F], dvar[R_F], df[R_F], dk[B(R_F)], noise partials[ceil(n / 256)].
 * Returns -2 (before any launch) for fidelity outside [0, 8), d outside [1, 8], M outside [1, 256], S < 1, n < 1 or
 * n S >= 2^31 - 32; mobo_acq_bwd_work_doubles returns 0 for those. */
size_t mobo_acq_bwd_work_doubles(int fidelity, int d, int M, int S, long long n);
int mobo_acq_moments_bwd(int fidelity, int d, int M, int S, long long n, const double* Zx,
                         const double* const* zf, const double* const* theta, const double* const* ops,
                         const double* const* samples, const double* raw_noise, double noise_lower,
                         double noise_upper, const double* X, const double* d_mu, const double* d_var,
                         int accumulate, double* dX, double* d_raw_noise, double* work, void* stream);
/* out[i] (+)=1/2 max(0, log vu[i] - log vc[i])   (_JES_MFDGP.forward, acquisition_functions/JESMOC_MFDGP.py:52) */
int mobo_jes(const double* var_uncond, const double* var_cond, long long n, int accumulate, double* out, void* stream);

/* ---- Pareto-sample generation (SURVEY.md section 8f-3) ----
 * Values (and optionally the x-gradient of the top layer) of the random-Fourier-feature function samples of an MFDGP
 * layer chain at n points: the closures returned by MFDGPHiddenLayer._sample_from_posterior(_layer0) /
 * _sample_from_prior(_layer0) (mobocmf/layers/mfdgp_hidden_layer.py:311-514) as MOOP evaluates them on its grid
 * (mobocmf/util/moop.py:221-286).  params[l] (device): layer 0 [W (F x d) | b (F) | theta (F)], layer >= 1
 * [W_x1 (F x d) | W_f (F) | W_x2 (F x d) | b_x1 (F) | b_x2 (F) | theta (3 F)].  scales (HOST, L x 3): layer 0
 * {sqrt(2 alpha / F), -, -}, layer >= 1 {sqrt(2 alpha_x1 / F) sqrt(nu_lin), sqrt(2 alpha_x1 alpha_f / F),
 * sqrt(2 alpha_x2 / F)}.  f: L x n (every layer's sample); grad: n x d or NULL.  L <= 4, d <= 8. */
int mobo_rff_eval(int L, int d, int F, const double* const* params, const double* scales, const double* x, long long n,
                  double* f, double* grad, void* stream);
/* mask[j] = 1 iff point j of pts (n x k, k <= 8, minimisation) is not dominated (MOOP.compute_pareto_front,
 * mobocmf/util/moop.py:141-185); of exact duplicates the lowest index survives. */
int mobo_pareto_mask(const double* pts, long long n, int k, unsigned char* mask, void* stream);

#ifdef __cplusplus
}
#endif
#endif
