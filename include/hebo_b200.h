/*
 * hebo_b200.h -- C ABI of libhebo_b200.so: the B200 (sm_100a) implementation of HEBO's
 * exact-GP fit + batched posterior/MACE hot path.
 *
 * This is the drop-in boundary a HEBO maintainer binds with ctypes (see INTEGRATION.md).
 * Every entry point cites the reference code it replaces (paths relative to the reference
 * checkout, HEBO/hebo/...).  The arithmetic the reference delegates to gpytorch
 * (Gram / Cholesky / solves / log-det / predictive variance; requirements.txt:6) is restated
 * in SURVEY.md Appendix A and implemented here from scratch.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no torch / C++ types cross the boundary.
 *   - Unless marked HOST, every pointer is a DEVICE pointer (tensor.data_ptr()).
 *   - fp32, row-major.  Square work matrices use the padded order NP = hb_padded_n(n)
 *     (next multiple of 128) with leading dimension NP; the pad is an identity block.
 *   - `stream` is a cudaStream_t passed as void* (torch.cuda.current_stream().cuda_stream).
 *   - The caller owns all memory, keeps it alive until the stream work completes; the
 *     library retains nothing between calls except lazily-built per-device state (kernel
 *     attributes, device-resident tile tables of the tensor-core fit stages, one capture stream).
 *   - Threading: like the reference (every call comes from the Python main thread,
 *     optimizers/hebo.py:143-186), one in-flight call per process and device; the lazily-built
 *     state is not guarded by locks.  hb_cholesky / hb_fit use a cooperative launch whose CTAs
 *     synchronise through flags in the caller's workspace: give concurrent calls distinct
 *     workspaces.
 *   - Return value: HB_OK, or an error below.  Never throws / aborts across the ABI.
 *     "Not positive definite" is reported through the device word `info` (LAPACK style:
 *     0 = ok, j>0 = leading minor j not PD) so the caller can reproduce the reference's
 *     jitter escalation (models/gp/gp.py:104-126, 140-157) without a CUDA error.
 *
 * Hyper-parameter vectors (P = d + 3 floats, gpytorch registration order, SURVEY Appendix A):
 *   raw[0] = raw_noise, raw[1] = mean constant, raw[2] = raw_outputscale, raw[3..3+d) = raw_lengthscale
 *   hyp[0] = sigma_n^2 = softplus(raw_noise)+noise_lb, hyp[1] = c, hyp[2] = s = softplus(raw_os),
 *   hyp[3..3+d) = lengthscale = softplus(raw_ls)
 *
 * Mixed numeric + categorical models and ard_kernel=False (the `_ex` entry points, hb_model_spec_t): the reference's
 * EmbTransform (models/layers.py:14-34: one nn.Embedding(num_uniq_c, emb_size_c) per categorical column, outputs
 * concatenated) feeds  ScaleKernel(Matern(ARD, numeric dims) * Matern-3/2(one lengthscale, embedding dims))
 * (models/gp/gp_util.py:39-59); the tables are trained inside the MLL.  Parameter order = module registration order:
 *   raw = (raw_noise, table_0 [num_uniq_0, emb_0] row-major, table_1, ..., [warp: raw_a[d], raw_b[d]], mean,
 *          raw_outputscale, raw_lengthscale[d if ard else 1] (absent when d = 0), raw_emb_lengthscale (when num_enum > 0))
 *   hyp = (sigma_n^2, c, s, lengthscale per numeric dim [d] (the shared one repeated when ard = 0), emb lengthscale,
 *          [warp: a[d], b[d] = 0.01 + 9.99 sigmoid(raw)])
 * With a warp the numeric features are z = (2 w(u) - 1) / l,  u = clamp((x~ + 1) / 2, 1e-6, 1 - 1e-6),  w = 1 - (1 - u^a)^b
 * (x~ = MinMax(-1,1)-scaled input); training rows are warped once per epoch (O(n d)), candidates inside the K* load stage.
 * hb_num_params() gives P.  Categories travel as int32 [rows, num_enum].
 */
#ifndef HEBO_B200_H
#define HEBO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HB_OK              0
#define HB_ERR_INVALID     1   /* bad argument (null pointer, size, unknown kernel id) */
#define HB_ERR_NOT_PD      2   /* host-visible "not positive definite" (hb_fit only)   */
#define HB_ERR_CUDA        3   /* CUDA runtime error; see hb_last_error()               */

#define HB_KERN_MATERN32   0   /* reference default: models/gp/gp_util.py:46 (nu = 1.5) */
#define HB_KERN_MATERN52   1   /* conf['kern'] injection, models/gp/gp.py:201            */
#define HB_KERN_RBF        2

/* Model description beyond the numeric ARD default (HOST struct; NULL = numeric-only, ard_kernel=True). */
typedef struct {
  int32_t        ard_kernel;  /* conf['ard_kernel'] (models/gp/gp.py:47, gp_util.py:45): 0 = one shared numeric lengthscale */
  int32_t        num_enum;    /* categorical columns e (0 = none)                                                          */
  const int32_t *num_uniqs;   /* HOST [e] categories per column (conf['num_uniqs'], optimizers/hebo.py:99-100)            */
  const int32_t *emb_sizes;   /* HOST [e] embedding widths (models/layers.py:19 default min(50, 1 + num_uniq // 2))       */
  int32_t        warp;        /* Kumaraswamy input warp of the numeric dims (BASELINE config 3; KumarWarp,
                                 models/nn/mono_layers/layers.py:85-117): 0 none, 1 exponents a, b LEARNED inside the MLL
                                 (2 d more parameters), 2 exponents fixed at the values in raw (never updated)             */
} hb_model_spec_t;

/* ---- library info (HOST) -------------------------------------------------------------- */
int32_t     hb_version(void);
const char *hb_last_error(void);                    /* last CUDA error string of this thread */
int64_t     hb_padded_n(int64_t n);                 /* NP: next multiple of 128               */
int32_t     hb_vnorm_operand_kind(void);            /* layout of hb_fit_state_t.Linv_hi/lo: 0 = two-level fp16 split (the only one built) */
/* Measurement hooks used by bench.py (HOST): number of kernels this library launched since the last reset, and
 * CUDA-event timing of the dominant kernel (the posterior variance contraction) on its launching stream. */
int64_t     hb_launch_count(int32_t reset);
int32_t     hb_profile_enable(int32_t on);
int32_t     hb_profile_collect(double *total_ms, int32_t *n_launches);
/* rows_flagged[0] = candidate rows that went through the tensor path since the last reset, [1] = how many of them the
 * precision guard re-contracted on the FP32 pipe (synchronises the device; current device only). */
int32_t     hb_guard_stats(uint64_t *rows_flagged, int32_t reset);
/* Workspace sizes in BYTES for the fused calls below. */
int64_t     hb_fit_workspace_bytes(int64_t n, int64_t d);
int64_t     hb_fit_workspace_bytes_ex(int64_t n, int64_t d, const hb_model_spec_t *spec);
int64_t     hb_num_params(int64_t d, const hb_model_spec_t *spec);      /* P: length of raw / grad / a Langevin row */
int64_t     hb_posterior_workspace_bytes(int64_t n, int64_t d, int64_t m_chunk);
int64_t     hb_pareto_workspace_bytes(int64_t m);

/* ---- hyper-parameter transform ---------------------------------------------------------
 * gpytorch Positive()/GreaterThan() constraints used at models/gp/gp.py:86 and
 * models/gp/gp_util.py:46,57: hyp = softplus(raw) (+ noise_lb for the noise). */
int32_t hb_transform_hypers(const float *raw, int64_t d, float noise_lb, float *hyp, void *stream);

/* ---- lengthscale initialisation  (models/gp/gp_util.py:47-52: per-dimension median of the pairwise |dx| over
 * <= 1000 rows, clamp >= 0.02) ------------------------------------------------------------------------------
 * Xt [d, NP] transposed scaled inputs; idx [d, k] int32 row subsets (np.random.choice per dimension) or NULL = rows
 * 0..k-1; k <= 1024.  out[d] = max(lower median of the k(k-1)/2 differences, clamp_min)  (torch.median semantics). */
int32_t hb_median_pdist(const float *Xt, int64_t n, int64_t d, const int32_t *idx, int64_t k, float clamp_min,
                        float *out, void *stream);

/* ---- Gram matrix  (replaces GPyTorchModel.forward -> self.cov(x_all), models/gp/gp.py:203-207,
 * kernel built at models/gp/gp_util.py:39-59) -----------------------------------------------
 * Xt       [d, NP] TRANSPOSED MinMax-scaled training inputs (column i = point i; pad columns ignored)
 * K        [NP, NP] out: lower triangle (incl. diagonal) of s*k(X,X) + (sigma_n^2 + jitter [+ noise_diag_i]) I;
 *          pad block = identity.  The strict upper triangle of off-diagonal tiles is not written.
 * noise_diag  [n] or NULL: per-row extra noise (BASELINE config 4 "heteroscedastic"; no reference). */
int32_t hb_gram(const float *Xt, int64_t n, int64_t d, const float *hyp, int32_t kern,
                const float *noise_diag, float jitter, float *K, void *stream);

/* ---- Cholesky  (replaces gpytorch psd_safe_cholesky inside ExactMarginalLogLikelihood /
 * the prediction strategy; call sites models/gp/gp.py:112-113, 148) ---------------------------
 * A [NP, NP] in/out, lower triangle; blocked right-looking, in place.  ws: >= 128*128*4 bytes.
 * info: device int32, set to j>0 if the leading minor j is not PD (left 0 otherwise; caller zeroes). */
int32_t hb_cholesky(float *A, int64_t np, float *ws, int32_t *info, void *stream);

/* ---- Triangular inverse and K^-1 (the n^3-class part of autograd's backward through the MLL,
 * models/gp/gp.py:115 loss.backward()) ---------------------------------------------------------
 * Linv = L^-1 (lower, strict upper zero-filled); tmp: [NP, NP] scratch.
 * Kinv = Linv^T Linv: lower tiles only. */
int32_t hb_tri_inverse(const float *L, int64_t np, float *Linv, float *tmp, void *stream);
int32_t hb_kinv(const float *Linv, int64_t np, float *Kinv, void *stream);

/* ---- alpha, quadratic form, log-det  (the data term of ExactMarginalLogLikelihood,
 * models/gp/gp.py:102,113; alpha is also the prediction-strategy mean cache, gp.py:148) --------
 * r = y - c (pad = 0).  alpha = Khat^-1 r, quad = r^T Khat^-1 r, logdet = 2 sum log L_ii.
 * scal[0] = quad, scal[1] = logdet (device, fp64 accumulated, stored as double[2]).
 * ws: >= 2*NP*sizeof(double) + 64*NP*sizeof(double). */
int32_t hb_solve_logdet(const float *L, const float *Linv, const float *y, int64_t n, int64_t np,
                        const float *hyp, float *alpha, double *scal, void *ws, void *stream);

/* ---- MLL gradient (closed form of SURVEY Appendix A; replaces loss.backward(), gp.py:115) ----
 * grad[P] = d(-mll/n)/d raw,  loss[0] = -mll/n including the Gamma(.5,.5) outputscale prior
 * (gp_util.py:57) and LogNormal(ln noise_guess, .5) noise prior (gp.py:87). */
int32_t hb_mll_grad(const float *Xt, int64_t n, int64_t d, const float *raw, const float *hyp,
                    int32_t kern, const float *Kinv, const float *alpha, const double *scal,
                    float noise_guess, float *grad, float *loss, void *ws, void *stream);

/* ---- pSGLD update  (models/nn/sgld.py:49-70 on torch.optim.RMSprop) --------------------------
 * xi: [P] N(0,1) draws or NULL (= pretrain phase, no Langevin noise). */
int32_t hb_psgld_step(float *raw, const float *grad, float *square_avg, int64_t p, float lr,
                      float rms_alpha, float rms_eps, float factor, const float *xi, void *stream);

/* ---- the whole fit loop  (GP.fit, models/gp/gp.py:96-135, optimizer='psgld') -----------------
 * Runs num_epochs x { transform, gram, cholesky, inverse, alpha/logdet, gradient, pSGLD } on
 * `stream` with one status read-back per epoch; on a not-PD epoch it retries with jitter x10 from
 * 1e-6 (fp32 value of gp.py:104-110) and gives up above 10 like gp.py:120-126.
 * langevin   [num_epochs, P] N(0,1) draws in registration order, or NULL for deterministic RMSprop.
 * losses     HOST [num_epochs] out (loss evaluated before each step), may be NULL.
 * After the loop it factorises at the final hypers and leaves in the workspace what predict needs;
 * hb_fit_state() returns the device pointers.  Returns HB_ERR_NOT_PD if the final factorisation fails. */
int32_t hb_fit(const float *Xt, const float *y, int64_t n, int64_t d, float *raw, int32_t kern,
               const float *noise_diag, float noise_lb, float noise_guess, float lr, int32_t num_epochs,
               const float *langevin, float *losses, void *ws, int64_t ws_bytes, void *stream);

/* Factorise at the hypers in `raw` and fill the predict state (used by hb_fit and by callers that
 * set hypers directly).  jitter_used HOST out (may be NULL). */
int32_t hb_factorize(const float *Xt, const float *y, int64_t n, int64_t d, const float *raw, int32_t kern,
                     const float *noise_diag, float noise_lb, float *jitter_used,
                     void *ws, int64_t ws_bytes, void *stream);

/* The general forms (mixed numeric + categorical inputs, ard_kernel=False; spec = NULL reduces to the calls above).
 * Xe DEVICE int32 [n, num_enum] training categories (NULL when num_enum = 0); Xt may be NULL when d = 0; raw [P] in the
 * order given at the top of this file; langevin [num_epochs, P]. */
int32_t hb_fit_ex(const float *Xt, const int32_t *Xe, const float *y, int64_t n, int64_t d, const hb_model_spec_t *spec,
                  float *raw, int32_t kern, const float *noise_diag, float noise_lb, float noise_guess, float lr,
                  int32_t num_epochs, const float *langevin, float *losses, void *ws, int64_t ws_bytes, void *stream);
int32_t hb_factorize_ex(const float *Xt, const int32_t *Xe, const float *y, int64_t n, int64_t d, const hb_model_spec_t *spec,
                        const float *raw, int32_t kern, const float *noise_diag, float noise_lb, float *jitter_used,
                        void *ws, int64_t ws_bytes, void *stream);
/* One MLL forward + backward at `raw` (closure of models/gp/gp.py:111-116: loss = -mll(gp(X)) ; loss.backward()):
 * grad [P], loss [1], info [1] (Cholesky status, LAPACK style) are DEVICE outputs; jitter is added to the diagonal. */
int32_t hb_mll_fwd_bwd(const float *Xt, const int32_t *Xe, const float *y, int64_t n, int64_t d, const hb_model_spec_t *spec,
                       const float *raw, int32_t kern, const float *noise_diag, float noise_lb, float noise_guess, float jitter,
                       float *grad, float *loss, int32_t *info, void *ws, int64_t ws_bytes, void *stream);

typedef struct {
  float  *hyp;     /* [H]        constrained hypers                       */
  float  *L;       /* [NP, NP]   Cholesky factor (lower)                   */
  float  *Linv;    /* [NP, NP]   L^-1 (lower)                              */
  float  *alpha;   /* [NP]       Khat^-1 (y - c), pad = 0                  */
  float  *Zt;      /* [d + De, NP] Xt / lengthscale (transposed), then the embedding features / their lengthscale */
  double *scal;    /* [2]        quad, logdet                              */
  float  *Linv_hi; /* [NP, NP] floats of storage: OPAQUE tensor-path operands of Linv.  Default (fp16 two-level split):  */
  float  *Linv_lo; /* h0 = rn_fp16(Linv*2^k) as NP*NP halfs in Linv_hi; h1 = rn_fp16((Linv*2^k - h0)*2048) as NP*NP halfs  */
                   /* in Linv_lo, followed by the float scale 2^k.  (hb_vnorm_operand_kind() == 0)                         */
  float  *tab_s;   /* [T] embedding tables / embedding lengthscale (mixed models; candidate side of the posterior)        */
  int32_t *emb_meta; /* OPAQUE categorical layout arrays (mixed models)                                                    */
  float  *grad;    /* [P] gradient of the last MLL evaluation             */
  float  *loss;    /* [1] loss of the last MLL evaluation                 */
} hb_fit_state_t;
int32_t hb_fit_state(void *ws, int64_t n, int64_t d, hb_fit_state_t *out);     /* HOST */
int32_t hb_fit_state_ex(void *ws, int64_t n, int64_t d, const hb_model_spec_t *spec, hb_fit_state_t *out);     /* HOST */

/* ---- fused posterior + MACE  (GP.predict, models/gp/gp.py:137-164, and MACE.eval,
 * acquisitions/acq.py:146-171; Mean/Sigma acq.py:66-82 read mu/var) ----------------------------
 * Xs        [m, d] RAW candidates; x_mul/x_add [d]: MinMax scale_/min_ (models/scalers.py:86-87)
 * Zt, alpha, Linv, hyp: from hb_fit_state.  Linv_hi/Linv_lo: from hb_fit_state -> variance contraction on the
 *           tcgen05 tensor cores (error-compensated fp16 two-level split, or 3xTF32); both NULL -> FP32 SIMT contraction.
 * y_mean,y_std: TorchStandardScaler (models/scalers.py:56-60).  pred_likeli: gp.py:158-159.
 * tau,kappa,eps: MACE(best_y, kappa, eps).  xi1, xi2 [m]: the two torch.randn draws of acq.py:154-155
 *           (NULL -> Philox N(0,1) from `seed`, independent streams per row).
 * F [m,3] out (LCB, -logEI, -logPI) or NULL; mu [m], var [m] out or NULL (original y units).
 * ws: hb_posterior_workspace_bytes(n, d, m_chunk); candidates are processed in chunks of m_chunk. */
int32_t hb_posterior_mace(const float *Xs, int64_t m, int64_t n, int64_t d,
                          const float *x_mul, const float *x_add,
                          const float *Zt, const float *alpha, const float *Linv,
                          const float *Linv_hi, const float *Linv_lo, const float *hyp, int32_t kern, float y_mean, float y_std, int32_t pred_likeli,
                          float tau, float kappa, float eps, const float *xi1, const float *xi2,
                          uint64_t seed, float *F, float *mu, float *var,
                          void *ws, int64_t ws_bytes, int64_t m_chunk, void *stream);

/* General form: Xe_s DEVICE int32 [m, num_enum] candidate categories, emb_meta / tab_s from hb_fit_state_ex
 * (all three NULL when num_enum = 0); Zt has d + De rows.  rng_offset: position of row 0 in the Philox stream (row r
 * draws the normals of stream position rng_offset + r), so a batch scored in several calls -- e.g. chunk by chunk while
 * the next chunk's host->device copy is in flight -- gets the same draws as one call over the whole batch. */
int32_t hb_posterior_mace_ex(const float *Xs, const int32_t *Xe_s, int64_t m, int64_t rng_offset, int64_t n, int64_t d,
                             const hb_model_spec_t *spec,
                             const int32_t *emb_meta, const float *tab_s, const float *x_mul, const float *x_add,
                             const float *Zt, const float *alpha, const float *Linv, const float *Linv_hi,
                             const float *Linv_lo, const float *hyp, int32_t kern, float y_mean, float y_std, int32_t pred_likeli,
                             float tau, float kappa, float eps, const float *xi1, const float *xi2, uint64_t seed, float *F,
                             float *mu, float *var, void *ws, int64_t ws_bytes, int64_t m_chunk, void *stream);

/* ---- GP.predict with gradients  (the `support_grad` contract: models/base_model.py:27-29 and
 * test/test_base_model.py:94-108 require predict() to be differentiable in Xc; gpytorch autograd through
 * models/gp/gp.py:137-164) -------------------------------------------------------------------------------------
 * Same inputs as hb_posterior_mace (FP32 SIMT contraction; Linv only).  mu, var [m] as above;
 * dmu, dvar [m, d] = d mu / d Xs, d var / d Xs (closed form; zero where a variance floor is active, like clamp_min).
 * ws: hb_posterior_workspace_bytes(n, d, m_chunk). */
int32_t hb_posterior_grad(const float *Xs, int64_t m, int64_t n, int64_t d,
                          const float *x_mul, const float *x_add,
                          const float *Zt, const float *alpha, const float *Linv, const float *hyp, int32_t kern,
                          float y_mean, float y_std, int32_t pred_likeli,
                          float *mu, float *var, float *dmu, float *dvar,
                          void *ws, int64_t ws_bytes, int64_t m_chunk, void *stream);

int32_t hb_posterior_grad_ex(const float *Xs, const int32_t *Xe_s, int64_t m, int64_t n, int64_t d, const hb_model_spec_t *spec,
                             const int32_t *emb_meta, const float *tab_s, const float *x_mul, const float *x_add,
                             const float *Zt, const float *alpha, const float *Linv, const float *hyp, int32_t kern, float y_mean,
                             float y_std, int32_t pred_likeli, float *mu, float *var, float *dmu, float *dvar, void *ws,
                             int64_t ws_bytes, int64_t m_chunk, void *stream);

/* ---- joint posterior samples  (GP.sample_y, models/gp/gp.py:166-177: pred.rsample(n_samples) of the [likelihood-]predictive
 * MultivariateNormal; used by NoisyAcq / GeneralBO, optimizers/general.py:131) ------------------------------------------
 * z [n_samples, m] N(0,1) draws (the caller's torch.randn, so the random stream stays the caller's); out [n_samples, m] in
 * original y units = (mu~ + R z) y_std + y_mean with R the Cholesky root of K** - V V^T (+ sigma_n^2 I with pred_likeli)
 * + jitter I, jitter from 1e-6 x10 per failed attempt (gpytorch psd_safe_cholesky, fp32); m <= 8192.  hyp_host: HOST copy of
 * hyp (noise / outputscale feed launch parameters).  Everything -- K*, K**, the rank-n update, the factorisation -- runs in
 * this library's kernels; the call synchronises once per factorisation attempt. */
int64_t hb_sample_workspace_bytes(int64_t n, int64_t d, const hb_model_spec_t *spec, int64_t m);
int32_t hb_sample_y(const float *Xs, const int32_t *Xe_s, int64_t m, int64_t n, int64_t d, const hb_model_spec_t *spec,
                    const int32_t *emb_meta, const float *tab_s, const float *x_mul, const float *x_add, const float *Zt,
                    const float *alpha, const float *Linv, const float *hyp, const float *hyp_host, int32_t kern, float y_mean,
                    float y_std, int32_t pred_likeli, const float *z, int32_t n_samples, float *out, float *jitter_used, void *ws,
                    int64_t ws_bytes, void *stream);

/* ---- MACE epilogue alone  (MACE.eval, acquisitions/acq.py:151-171, over any model's predict output) ----
 * mu, var [m] in original y units (device); noise_var = model.noise (gp.py:182-184); xi1/xi2 as above.
 * F [m,3] out = (LCB, -logEI, -logPI). */
int32_t hb_mace_epilogue(const float *mu, const float *var, int64_t m, float noise_var, float tau, float kappa,
                         float eps, const float *xi1, const float *xi2, uint64_t seed, float *F, void *stream);

/* ---- GeneralAcq epilogue  (GeneralAcq.eval, acquisitions/acq.py:233-242, over any multi-output model's predict output;
 * the acquisition of GeneralBO, optimizers/general.py:23-204) -------------------------------------------------------------
 * mu, var [O, m] output-major, O = num_obj + num_constr (O calls of hb_posterior_mace_ex with F = NULL write one row each),
 * original y units; noise_var [O] device (model.noise, read when use_noise); xi [m, O] the reference's one torch.randn(py.shape)
 * draw, or NULL -> Philox N(0,1) keyed by (seed, rng_offset + row, output).
 * out [m, O] = py (+ sqrt(noise) xi) - kappa ps (objective columns) | - c_kappa ps (constraint columns), ps = max(sqrt(ps2), eps);
 * cv [m] out or NULL: sum_j max(0, out[:, num_obj + j]), the constraint violation of evolution_optimizer.py:104-105 (F / G).
 * 1 <= num_obj <= 8, num_obj + num_constr <= 64.  One launch, no host synchronisation. */
int32_t hb_general_acq_epilogue(const float *mu, const float *var, int64_t m, int32_t num_obj, int32_t num_constr,
                                const float *noise_var, float kappa, float c_kappa, int32_t use_noise, const float *xi, uint64_t seed,
                                int64_t rng_offset, float *out, float *cv, void *stream);

/* ---- K-objective constrained non-dominated filter  (the rank-0 / feasible set NSGA-II returns as res.X,
 * acq_optimizers/evolution_optimizer.py:135-149, and GeneralBO's front, optimizers/general.py:182-195) --------------------
 * F [m, ldf] (objective columns 0..K-1 of each row, ldf >= K, 1 <= K <= 8); cv [m] or NULL.  idx_out [m] int32 ascending
 * indices of the non-dominated FEASIBLE rows (cv <= 0); count device int32.  Rows with a NaN objective or cv are excluded.
 * If no row is feasible the result is the one row of least cv (lowest index on ties).  ws: hb_pareto_workspace_bytes(m),
 * enough for every K.  No host synchronisation. */
int32_t hb_pareto_front(const float *F, int64_t m, int32_t K, int64_t ldf, const float *cv, int32_t *idx_out, int32_t *count,
                        void *ws, int64_t ws_bytes, void *stream);

/* ---- 3-objective non-dominated filter  (the rank-0 set NSGA-II returns as res.X,
 * acq_optimizers/evolution_optimizer.py:141-149) ----------------------------------------------
 * F [m,3]; idx_out [m] int32 ascending indices of the non-dominated rows; count device int32.
 * Rows with a NaN objective are excluded (they can neither dominate nor be dominated, and must never be recommended). */
int32_t hb_pareto_front3(const float *F, int64_t m, int32_t *idx_out, int32_t *count,
                         void *ws, int64_t ws_bytes, void *stream);

/* ---- device NSGA-II  (acq_optimizers/evolution_optimizer.py:107-160: pymoo NSGA2 with MixedVariableMating over the MACE
 * objectives; variable typing :26-41).  The population lives on the device: X [pop, D] fp32 rows in the optimisation space
 * (d numeric columns, then D - d categorical indices), kind [D] (0 Real, 1 Integer, 2 Choice), lb / ub [D],
 * fixed [D] (NaN = free; otherwise the value of a fix_input column, :97-101).  Every call also emits the rows split into
 * the model's inputs Xc [pop, d] fp32 / Xe [pop, D - d] int32.  One generation = hb_nsga2_mate -> hb_posterior_mace_ex on
 * the offspring -> hb_nsga2_survive (rank + crowding of the 2 pop merged rows, duplicates and non-finite objectives never
 * survive; pop <= 256); nothing synchronises with the host.  Philox streams keyed by (seed, generation). */
int32_t hb_nsga2_init(float *X, int64_t pop, int64_t D, int64_t d, const int32_t *kind, const float *lb, const float *ub,
                      const float *fixed, const float *init, int64_t n_init, uint64_t seed, float *Xc, int32_t *Xe, void *stream);
int32_t hb_nsga2_mate(const float *X, int64_t pop, int64_t D, int64_t d, const int32_t *kind, const float *lb, const float *ub,
                      const float *fixed, uint64_t seed, int32_t generation, float *C, float *Cc, int32_t *Ce, void *stream);
int32_t hb_nsga2_survive(const float *X, const float *F, const float *C, const float *FC, int64_t pop, int64_t D, int64_t d,
                         float *X_next, float *F_next, float *Xc_next, int32_t *Xe_next, void *stream);

/* K-objective survival with constraints (evolution_optimizer.py:104-105 hands pymoo F [pop, K] and G; the survival replaces
 * pymoo's rank-and-crowding with its filter_infeasible rule): F / FC [pop, K], CV / CVC [pop] constraint violations (both
 * NULL = unconstrained).  Feasible rows (cv <= 0) go through rank-and-crowding for min(n_feasible, pop) slots; the rest go to
 * the other rows in ascending cv (lower merged index first); duplicates and non-finite objectives only fill slots nothing
 * else can.  Survivors in ascending merged-row order; CV_next [pop] required with CV.  1 <= K <= 8.
 * hb_nsga2_survive == K = 3 without constraints. */
int32_t hb_nsga2_survive_k(const float *X, const float *F, const float *CV, const float *C, const float *FC, const float *CVC,
                           int64_t pop, int64_t D, int64_t d, int32_t K, float *X_next, float *F_next, float *CV_next,
                           float *Xc_next, int32_t *Xe_next, void *stream);

/* ---- multi-GPU front exchange  (candidate-sharded scoring, BASELINE config 5: every rank filters its shard, ONE
 * all-gather of fixed-capacity front buffers, every rank merges; no reference counterpart -- the reference is one process,
 * optimizers/hebo.py:119-194) ------------------------------------------------------------------------------------
 * Buffer layout [(capacity + 1), 8] fp32: row 0 = (count, overflow flag, 0...); row 1 + j = (F0, F1, F2, mu, sigma,
 * id_lo, id_hi, 0) with the global candidate id = id_lo + 2^24 id_hi; unused rows hold +inf objectives.
 * hb_front_pack : F [m,3], mu / var [m] (or NULL), idx / count from hb_pareto_front3, row_offset = first global id of
 *                 this shard -> out.  A front larger than `capacity` sets the overflow flag (never silently truncated).
 * hb_front_merge: all_buf [world][capacity + 1][8] (the all-gathered buffers) -> out [(world * capacity + 1), 8]: the
 *                 non-dominated rows of the union in ascending global-id order.  No host synchronisation in either call. */
int64_t hb_front_merge_workspace_bytes(int64_t world, int64_t capacity);
int32_t hb_front_pack(const float *F, const float *mu, const float *var, const int32_t *idx, const int32_t *count,
                      int64_t row_offset, int64_t capacity, float *out, void *stream);
int32_t hb_front_merge(const float *all_buf, int64_t world, int64_t capacity, float *out, void *ws, int64_t ws_bytes,
                       void *stream);

#ifdef __cplusplus
}
#endif
#endif /* HEBO_B200_H */
