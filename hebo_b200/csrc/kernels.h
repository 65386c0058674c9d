// Internal launcher declarations (C++ linkage); the C ABI lives in api.cu / include/hebo_b200.h.
#pragma once
#include <cuda_fp16.h>
#include "common.cuh"

namespace hb {

// hi/lo (3xTF32) companion buffers of the fit's tensor-core path (fit_tc.cu); all [NP, NP] except P [NP, 512]
struct TcBuffers {
  float *L_hi, *L_lo, *Linv_hi, *Linv_lo, *U_hi, *U_lo, *T_hi, *T_lo, *P_hi, *P_lo;
};

// Parameter layout of the (optionally mixed numeric + categorical) exact GP, in the reference's registration order
// (likelihood.raw_noise, embedding tables, mean constant, raw_outputscale, numeric raw_lengthscale[s], embedding
// raw_lengthscale: HEBO/hebo/models/gp/gp.py:86-103, gp_util.py:22-59, layers.py:14-34).  With e == 0 and ard == 1 this is
// the numeric-only layout raw = (noise, mean, outputscale, lengthscale[d]).
//   raw : [P]  P = 3 + T + 2 d [warp] + n_ls + (e > 0):  noise, tables, warp a / b (feature-extractor parameters), mean,
//              outputscale, numeric lengthscale(s), embedding lengthscale
//   hyp : [H]  H = 3 + d + (e > 0) + 2 d [warp]:  sigma_n^2, c, s, lengthscale per numeric dim (expanded when ard == 0),
//              emb lengthscale, Kumaraswamy exponents a[d], b[d]
struct ModelSpec {
  int d = 0;      // numeric dims (0 allowed when e > 0)
  int ard = 1;    // conf['ard_kernel'] (gp.py:47)
  int e = 0;      // categorical columns
  int De = 0;     // total embedding width  sum_c emb_size_c
  int T = 0;      // total table entries    sum_c num_uniq_c * emb_size_c
  int warp = 0;   // Kumaraswamy input warp of the numeric dims: 0 none, 1 learned exponents a, b (2 d parameters), 2 frozen
  // device int32 arrays living in the fit workspace (nullptr when e == 0)
  const int32_t *q_col = nullptr, *q_loc = nullptr;               // [De] categorical column / coordinate inside it
  const int32_t *tab_off = nullptr, *emb_size = nullptr;          // [e]  offset of table c inside the T block, its width
  const int32_t *ent_col = nullptr, *ent_u = nullptr, *ent_q = nullptr;   // [T] (column, category, coordinate) of entry t
  const int32_t *Xe = nullptr;                                    // [n, e] training categories
  __host__ __device__ int n_ls() const { return d == 0 ? 0 : (ard ? d : 1); }
  __host__ __device__ int i_tab() const { return 1; }
  __host__ __device__ int n_w() const { return warp ? 2 * d : 0; }       // raw warp parameters (a[d], b[d]) after the tables
  __host__ __device__ int i_wa() const { return 1 + T; }
  __host__ __device__ int i_wb() const { return 1 + T + d; }
  __host__ __device__ int i_mean() const { return 1 + T + n_w(); }
  __host__ __device__ int i_os() const { return 2 + T + n_w(); }
  __host__ __device__ int i_ls() const { return 3 + T + n_w(); }
  __host__ __device__ int i_le() const { return 3 + T + n_w() + n_ls(); }
  __host__ __device__ int P() const { return 3 + T + n_w() + n_ls() + (e > 0 ? 1 : 0); }
  __host__ __device__ int h_wa() const { return 3 + d + (e > 0 ? 1 : 0); }        // hyp: a[d], b[d] after the lengthscales
  __host__ __device__ int h_wb() const { return h_wa() + d; }
  __host__ __device__ int H() const { return 3 + d + (e > 0 ? 1 : 0) + n_w(); }
  __host__ __device__ int dtot() const { return d + De; }
};

// cholesky.cu / linalg.cu   (tc == nullptr -> FP32 SIMT everywhere)
int launch_cholesky(float *A, int64_t np, float *ws, int32_t *info, cudaStream_t st, const TcBuffers *tc = nullptr);
// fit_tc.cu
int launch_triinv_base2(const float *L, int64_t np, float *Linv, float *Linv_hi, float *Linv_lo, float *U_hi, float *U_lo,
                        cudaStream_t st);
void chol_timer_mark(int cls, cudaStream_t st);   // debug timing (HEBO_B200_CHOL_TIMING=1)
int launch_chol_outer_update_tc(float *A, int64_t np, int64_t cb, int64_t ce, const TcBuffers &tc, cudaStream_t st);
int launch_tri_inverse_tc(const float *L, int64_t np, float *Linv, const TcBuffers &tc, bool zero_fill, cudaStream_t st);
int launch_kinv_tc(int64_t np, float *Kinv, const TcBuffers &tc, cudaStream_t st);
int launch_tri_inverse(const float *L, int64_t np, float *Linv, float *tmp, cudaStream_t st);
int launch_kinv(const float *Linv, int64_t np, float *Kinv, cudaStream_t st);
int launch_linv_refine(float *L, float *Linv, int64_t np, float *R, float *out, cudaStream_t st);
int launch_solve_logdet(const float *L, const float *Linv, const float *y, int64_t n, int64_t np,
                        const float *hyp, float *alpha, double *scal, void *ws, cudaStream_t st);
size_t solve_ws_bytes(int64_t np);

// pairwise.cu
int launch_transform_hypers(const float *raw, const ModelSpec &sp, float noise_lb, float *hyp, cudaStream_t st);
int launch_gram(const float *Xt, const float *Ets, int64_t n, int64_t np, const ModelSpec &sp, const float *hyp, int kern,
                const float *noise_diag, float jitter, float *K, cudaStream_t st);
int launch_mll_grad(const float *Xt, const float *Ets, int64_t n, int64_t np, const ModelSpec &sp, const float *raw,
                    const float *hyp, int kern, const float *Kinv, const float *alpha, const double *scal, float noise_guess,
                    float *grad, float *loss, void *ws, cudaStream_t st, const float *dZa = nullptr, const float *dZb = nullptr);
size_t grad_ws_bytes(int64_t np, const ModelSpec &sp);
int launch_emb_gather(const float *tables, const ModelSpec &sp, int64_t n, int64_t np, const float *hyp, float *Ets, float *tab_s,
                      cudaStream_t st);
int launch_psgld(float *raw, const float *grad, float *sq, int64_t p, float lr, float a, float eps,
                 float factor, const float *xi, cudaStream_t st);
int launch_scale_zt(const float *Xt, int64_t np, const ModelSpec &sp, const float *hyp, float *Zt, float *dZa, float *dZb,
                    cudaStream_t st);

// init.cu
int launch_median_pdist(const float *Xt, int64_t np, int64_t d, const int32_t *idx, int64_t k, float clamp_min,
                        float *out, cudaStream_t st);

// posterior.cu
int launch_posterior_mace(const float *Xs, const int32_t *Xe_s, int64_t m, int64_t rng_offset, int64_t n, int64_t np, const ModelSpec &sp,
                          const float *tab_s, const float *x_mul,
                          const float *x_add, const float *Zt, const float *alpha, const float *Linv,
                          const float *Linv_hi, const float *Linv_lo, const float *hyp, int kern, float y_mean, float y_std, int pred_likeli, float tau,
                          float kappa, float eps, const float *xi1, const float *xi2, uint64_t seed, float *F,
                          float *mu, float *var, void *ws, int64_t ws_bytes, int64_t m_chunk, cudaStream_t st);
size_t posterior_ws_bytes(int64_t np, int64_t d, int64_t m_chunk);
int guard_stats(unsigned long long *out, int reset);
int launch_mace_only(const float *mu, const float *var, int64_t m, float noise_var, float tau, float kappa, float eps,
                     const float *xi1, const float *xi2, uint64_t seed, float *F, cudaStream_t st);
int launch_general_acq(const float *mu, const float *var, int64_t m, int num_obj, int num_constr, const float *noise_var,
                       float kappa, float c_kappa, int use_noise, const float *xi, uint64_t seed, int64_t rng_offset, float *out,
                       float *cv, cudaStream_t st);

// fp16 two-level split tensor path of the posterior (vnorm_h16.cu: tcgen05 / TMEM / TMA)
int kstar_groups(int64_t np);
int launch_kstar_plain(const float *xs, const int32_t *xe, int64_t mc, const ModelSpec &sp, const float *tab_s,
                       const float *x_mul, const float *x_add, const float *Zt,
                       const float *alpha, const float *hyp, int64_t n, int64_t np, int kern, float *KS, float *mupart,
                       int64_t mc_pad, cudaStream_t st);
int launch_posterior_grad(const float *Xs, const int32_t *Xe_s, int64_t m, int64_t n, int64_t np, const ModelSpec &sp,
                          const float *tab_s, const float *x_mul, const float *x_add,
                          const float *Zt, const float *alpha, const float *Linv, const float *hyp, int kern, float y_mean,
                          float y_std, int pred_likeli, float *mu, float *var, float *dmu, float *dvar, void *ws,
                          int64_t ws_bytes, int64_t m_chunk, cudaStream_t st);
int launch_split_h16(const float *x, int64_t count, __half *h0, __half *h1, float *scale_slot, cudaStream_t st);
int launch_vnorm_h16(const __half *ks_h0, const __half *ks_h1, int64_t ks_rows, const __half *linv_h0, const __half *linv_h1,
                     const float *scale_b, const float *hyp, int64_t np, int64_t mc_pad, int64_t vpart_stride, float *vpart,
                     cudaStream_t st);

// pareto.cu
int launch_pareto(const float *F, int64_t m, int K, int64_t ldf, const float *cv, int32_t *idx_out, int32_t *count, void *ws,
                  int64_t ws_bytes, cudaStream_t st);
int launch_pareto3(const float *F, int64_t m, int32_t *idx_out, int32_t *count, void *ws, int64_t ws_bytes,
                   cudaStream_t st);
size_t pareto_ws_bytes(int64_t m);
int launch_front_pack(const float *F, const float *mu, const float *var, const int32_t *idx, const int32_t *count,
                      int64_t row_offset, int64_t capacity, float *out, cudaStream_t st);
size_t front_merge_ws_bytes(int64_t world, int64_t capacity);
int launch_front_merge(const float *all, int64_t world, int64_t capacity, float *out, void *ws, int64_t ws_bytes,
                       cudaStream_t st);

size_t sample_ws_bytes(int64_t np, int64_t dtot, int64_t m);
int launch_sample_y(const float *Xs, const int32_t *Xe_s, int64_t m, int64_t n, int64_t np, const ModelSpec &sp, const float *tab_s,
                    const float *x_mul, const float *x_add, const float *Zt, const float *alpha, const float *Linv, const float *hyp,
                    const float *hyp_host, int kern, float y_mean, float y_std, int pred_likeli, const float *z, int n_samples,
                    float *out, float *jitter_used, void *ws, int64_t ws_bytes, cudaStream_t st);
// nsga.cu
int launch_nsga_init(float *X, int64_t P, int64_t D, int64_t d, const int32_t *kind, const float *lb, const float *ub,
                     const float *fixed, const float *init, int64_t n_init, uint64_t seed, float *Xc, int32_t *Xe, cudaStream_t st);
int launch_nsga_mate(const float *X, int64_t P, int64_t D, int64_t d, const int32_t *kind, const float *lb, const float *ub,
                     const float *fixed, uint64_t seed, int gen, float *C, float *Cc, int32_t *Ce, cudaStream_t st);
int launch_nsga_survive(const float *X, const float *F, const float *C, const float *FC, int64_t P, int64_t D, int64_t d,
                        float *Xn, float *Fn, float *Xcn, int32_t *Xen, cudaStream_t st);
int launch_nsga_survive_k(const float *X, const float *F, const float *CV, const float *C, const float *FC, const float *CVC,
                          int64_t P, int64_t D, int64_t d, int K, float *Xn, float *Fn, float *CVn, float *Xcn, int32_t *Xen,
                          cudaStream_t st);

}  // namespace hb
