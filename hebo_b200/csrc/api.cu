// extern "C" entry points of libhebo_b200.so (declared in include/hebo_b200.h) and the native fit-loop
// runtime (the 100-epoch pSGLD loop of HEBO/hebo/models/gp/gp.py:96-135 without Python in the loop).
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <vector>

#include "h16.cuh"
#include "kernels.h"

namespace hb {

static thread_local char g_err[512] = "";

void set_error(cudaError_t e, const char *where) {
  snprintf(g_err, sizeof(g_err), "%s: %s", where, cudaGetErrorString(e));
}

int check_launch(const char *where) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error(e, where);
    return HB_ERR_CUDA;
  }
  return HB_OK;
}

static std::atomic<long long> g_launches{0};
void count_launches(int n) { g_launches += n; }

// CUDA-event brackets around the dominant kernel (posterior variance contraction), recorded on the launching
// stream; enabled by bench.py through hb_profile_enable and read back with hb_profile_collect.
struct Prof {
  bool on = false;
  std::vector<cudaEvent_t> a, b;
  size_t used = 0;
};
static Prof g_prof;
void prof_begin(cudaStream_t st) {
  if (!g_prof.on) return;
  if (g_prof.used == g_prof.a.size()) {
    cudaEvent_t e0, e1;
    if (cudaEventCreate(&e0) != cudaSuccess || cudaEventCreate(&e1) != cudaSuccess) return;
    g_prof.a.push_back(e0);
    g_prof.b.push_back(e1);
  }
  cudaEventRecord(g_prof.a[g_prof.used], st);
}
void prof_end(cudaStream_t st) {
  if (!g_prof.on || g_prof.used >= g_prof.a.size()) return;
  cudaEventRecord(g_prof.b[g_prof.used], st);
  g_prof.used++;
}

// ---------------------------------------------------------------- fit workspace layout
constexpr int FIT_BATCH = 16;   // epochs replayed per host synchronisation (CUDA-graph fit loop)

struct FitWs {
  float *hyp, *grad, *sq, *loss;
  int32_t *info;          // [0] factorisation status, [1] epoch counter, [2] replay slot of the current batch
  double *scal;
  float *status;          // [FIT_BATCH][2]: (info, loss) of every epoch of a batch
  float *L, *Linv, *tmp, *alpha, *Zt, *cholws, *Linv_hi, *Linv_lo;
  float *Ets;             // = Zt + d * NP: embedding rows of the scaled feature matrix (mixed model)
  float *dZa, *dZb;       // [d, NP] d Zt / d a_k, d Zt / d b_k (warped model)
  float *tab_s;           // [T] embedding tables / embedding lengthscale (candidate side of the posterior)
  int32_t *meta, *Xe;     // categorical layout arrays (ModelSpec) and the training categories [n, e]
  TcBuffers tc;
  void *solvews, *gradws;
  size_t total;
};

static inline size_t al256(size_t x) { return (x + 255) / 256 * 256; }

// ---- ModelSpec from the C-ABI description; device arrays bound separately (they live in the fit workspace)
static bool build_spec(int64_t d, const hb_model_spec_t *c, ModelSpec &sp) {
  sp = ModelSpec();
  if (d < 0) return false;
  sp.d = (int)d;
  if (c) {
    sp.ard = c->ard_kernel ? 1 : 0;
    sp.warp = (sp.d > 0) ? c->warp : 0;
    if (sp.warp < 0 || sp.warp > 2) return false;
    sp.e = c->num_enum;
    if (sp.e < 0 || (sp.e > 0 && (!c->num_uniqs || !c->emb_sizes))) return false;
    for (int k = 0; k < sp.e; ++k) {
      if (c->num_uniqs[k] <= 0 || c->emb_sizes[k] <= 0) return false;
      sp.De += c->emb_sizes[k];
      sp.T += c->num_uniqs[k] * c->emb_sizes[k];
    }
  }
  return sp.dtot() > 0;
}
static size_t meta_ints(const ModelSpec &sp) { return (size_t)2 * sp.De + 2 * sp.e + 3 * sp.T; }
static void bind_meta(ModelSpec &sp, const int32_t *meta, const int32_t *Xe) {
  if (sp.e <= 0) return;
  sp.q_col = meta;
  sp.q_loc = sp.q_col + sp.De;
  sp.tab_off = sp.q_loc + sp.De;
  sp.emb_size = sp.tab_off + sp.e;
  sp.ent_col = sp.emb_size + sp.e;
  sp.ent_u = sp.ent_col + sp.T;
  sp.ent_q = sp.ent_u + sp.T;
  sp.Xe = Xe;
}
static void fill_meta_host(const hb_model_spec_t *c, const ModelSpec &sp, std::vector<int32_t> &m) {
  m.assign(meta_ints(sp), 0);
  int32_t *q_col = m.data(), *q_loc = q_col + sp.De, *tab_off = q_loc + sp.De, *emb_size = tab_off + sp.e;
  int32_t *ent_col = emb_size + sp.e, *ent_u = ent_col + sp.T, *ent_q = ent_u + sp.T;
  int q = 0, t = 0;
  for (int k = 0; k < sp.e; ++k) {
    tab_off[k] = t;
    emb_size[k] = c->emb_sizes[k];
    for (int j = 0; j < c->emb_sizes[k]; ++j, ++q) {
      q_col[q] = k;
      q_loc[q] = j;
    }
    for (int u = 0; u < c->num_uniqs[k]; ++u)
      for (int j = 0; j < c->emb_sizes[k]; ++j, ++t) {   // nn.Embedding weight [num_uniq, emb_size], row-major
        ent_col[t] = k;
        ent_u[t] = u;
        ent_q[t] = j;
      }
  }
}

static FitWs carve_fit(void *base, int64_t n, const ModelSpec &sp) {
  const int64_t np = round_up(n, TILE);
  const int64_t P = sp.P(), H = sp.H();
  unsigned char *p = reinterpret_cast<unsigned char *>(base);
  size_t off = 0;
  FitWs w;
  auto take = [&](size_t bytes) {
    void *r = p ? (void *)(p + off) : nullptr;
    off += al256(bytes);
    return r;
  };
  w.hyp = (float *)take(H * 4);
  w.grad = (float *)take(P * 4);
  w.sq = (float *)take(P * 4);
  w.loss = (float *)take(16);
  w.info = (int32_t *)take(16);
  w.scal = (double *)take(16);
  w.status = (float *)take(FIT_BATCH * 2 * sizeof(float));
  w.L = (float *)take((size_t)np * np * 4);
  w.Linv = (float *)take((size_t)np * np * 4);
  w.tmp = (float *)take((size_t)np * np * 4);
  w.Linv_hi = (float *)take((size_t)np * np * 4);
  w.Linv_lo = (float *)take((size_t)np * np * 4);
  w.tc.Linv_hi = w.Linv_hi;
  w.tc.Linv_lo = w.Linv_lo;
  w.tc.L_hi = (float *)take((size_t)np * np * 4);
  w.tc.L_lo = (float *)take((size_t)np * np * 4);
  w.tc.U_hi = (float *)take((size_t)np * np * 4);
  w.tc.U_lo = (float *)take((size_t)np * np * 4);
  w.tc.T_hi = (float *)take((size_t)np * np * 4);
  w.tc.T_lo = (float *)take((size_t)np * np * 4);
  w.tc.P_hi = (float *)take((size_t)np * 512 * 4);
  w.tc.P_lo = (float *)take((size_t)np * 512 * 4);
  w.alpha = (float *)take((size_t)np * 4);
  w.Zt = (float *)take((size_t)sp.dtot() * np * 4);
  w.Ets = w.Zt ? w.Zt + (size_t)sp.d * np : nullptr;
  w.dZa = (float *)take(sp.warp ? (size_t)sp.d * np * 4 : 16);
  w.dZb = (float *)take(sp.warp ? (size_t)sp.d * np * 4 : 16);
  w.cholws = (float *)take((size_t)TILE * TILE * 4);
  w.solvews = take(solve_ws_bytes(np));
  w.gradws = take(grad_ws_bytes(np, sp));
  w.tab_s = (float *)take((size_t)(sp.T > 0 ? sp.T : 1) * 4);
  w.meta = (int32_t *)take((meta_ints(sp) + 1) * 4);
  w.Xe = (int32_t *)take(((size_t)n * sp.e + 1) * 4);
  w.total = off;
  return w;
}

struct HostStatus {
  int32_t info;
  float loss;
  int32_t set_epoch;
  int32_t pad;
  float batch[FIT_BATCH * 2];   // (info as float bits, loss) per replay slot
};
// one pinned status block per DEVICE (the header allows one in-flight call per process and device)
static HostStatus *pinned_status() {
  static HostStatus *p[MAX_DEVICES] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= MAX_DEVICES) return nullptr;
  if (!p[dev]) {
    if (cudaMallocHost(&p[dev], sizeof(HostStatus)) != cudaSuccess) p[dev] = nullptr;
  }
  return p[dev];
}

// conditional pSGLD (sgld.py:57-70): skipped on the device when the epoch's factorisation failed.  One block.  The epoch
// index lives on the device (info[1], advanced on success only), so the same launch -- and a CUDA graph replay of it -- works
// for every epoch: the Langevin row is langevin[epoch] once epoch + 1 > pretrain (n_step is incremented first in the
// reference).  (info, loss) of the attempt go to status[slot], slot = info[2]++.
__global__ void __launch_bounds__(256) psgld_guarded_kernel(float *__restrict__ raw, const float *__restrict__ grad,
                                                            float *__restrict__ sq, int p, float lr, float a, float eps,
                                                            float factor, const float *__restrict__ langevin, int pretrain,
                                                            int32_t *__restrict__ info, const float *__restrict__ loss,
                                                            float *__restrict__ status, const float *__restrict__ hyp,
                                                            int nhyp, int frozen_begin, int frozen_end) {
  // hopeless epoch: a constrained hyper-parameter is not finite or a lengthscale / outputscale has underflowed to zero
  // (pSGLD's Langevin step divides by sqrt(sqrt(v) + 1e-8): a parameter with a vanishing gradient random-walks in steps of
  // ~5 raw units, sgld.py:64-70).  K is then NaN, no jitter can repair it, and -- as in the reference, where the closure
  // raises before the optimiser updates anything (gp.py:111-126) -- no later epoch can change the parameters: status -1.
  __shared__ int bad;
  if (threadIdx.x == 0) bad = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < nhyp; i += blockDim.x) {
    const float h = hyp[i];
    if (!isfinite(h) || (i != 1 && !(h > 0.0f))) bad = 1;
  }
  __syncthreads();
  const int ok = info[0] == 0 && !bad, ep = info[1], slot = info[2];
  const float *xi = (langevin && (ep + 1) > pretrain) ? langevin + (int64_t)ep * p : nullptr;
  if (ok) {
    for (int i = threadIdx.x; i < p; i += blockDim.x) {
      if (i >= frozen_begin && i < frozen_end) continue;   // fixed (not learned) warp exponents are not optimiser parameters
      const float g = grad[i];
      const float v = a * sq[i] + (1.0f - a) * g * g;
      sq[i] = v;
      const float avg = sqrtf(v) + eps;
      float x = raw[i] - lr * g / avg;
      if (xi) x += factor * sqrtf(2.0f * lr / avg) * xi[i];
      raw[i] = x;
    }
  }
  __syncthreads();   // every thread has read the counters
  if (threadIdx.x == 0) {
    if (slot < FIT_BATCH) {
      status[2 * slot + 0] = __int_as_float(bad ? -1 : info[0]);
      status[2 * slot + 1] = loss[0];
    }
    info[2] = slot + 1;
    if (ok) info[1] = ep + 1;
  }
}

// gram -> cholesky at (hyp, jitter); info left on the device
// FP32 SIMT fallback for the fit's GEMM stages: HEBO_B200_FIT_SIMT=1 (A/B timing, debugging)
static bool fit_use_tc() {
  static int v = -1;
  if (v < 0) {
    const char *e = getenv("HEBO_B200_FIT_SIMT");
    v = (e && e[0] == '1') ? 0 : 1;
  }
  return v == 1;
}

// (mixed model: gathers the embedding features at the current tables / lengthscale first)
static int factor_once(const float *Xt, int64_t n, int64_t np, const ModelSpec &sp, const float *raw, int kern,
                       const float *noise_diag, float jitter, FitWs &w, cudaStream_t st, bool allow_tc = true) {
  HB_CUDA(cudaMemsetAsync(w.info, 0, sizeof(int32_t), st));
  int s = launch_emb_gather(raw + sp.i_tab(), sp, n, np, w.hyp, w.Ets, w.tab_s, st);
  if (s != HB_OK) return s;
  if (sp.warp) {   // warped features (and their exponent derivatives) at the current a, b, lengthscales
    s = launch_scale_zt(Xt, np, sp, w.hyp, w.Zt, w.dZa, w.dZb, st);
    if (s != HB_OK) return s;
  }
  s = launch_gram(sp.warp ? w.Zt : Xt, w.Ets, n, np, sp, w.hyp, kern, noise_diag, jitter, w.L, st);
  if (s != HB_OK) return s;
  return launch_cholesky(w.L, np, w.cholws, w.info, st, (allow_tc && fit_use_tc()) ? &w.tc : nullptr);
}

static float next_jitter(float j) { return j == 0.0f ? 1e-6f : j * 10.0f; }   // fp32 ladder of gp.py:104-110
constexpr float JITTER_MAX = 1e3f;                                             // 100 * (jitter <= 10), gp.py:121

}  // namespace hb

using namespace hb;

extern "C" {

int32_t hb_version(void) { return 200; }
const char *hb_last_error(void) { return g_err; }
int64_t hb_padded_n(int64_t n) { return round_up(n, TILE); }
int32_t hb_vnorm_operand_kind(void) { return 0; }

int64_t hb_launch_count(int32_t reset) {
  long long v = g_launches.load();
  if (reset) g_launches = 0;
  return (int64_t)v;
}

int32_t hb_profile_enable(int32_t on) {
  g_prof.on = on != 0;
  g_prof.used = 0;
  return HB_OK;
}

int32_t hb_profile_collect(double *total_ms, int32_t *n_launches) {
  if (!total_ms || !n_launches) return HB_ERR_INVALID;
  double tot = 0.0;
  for (size_t i = 0; i < g_prof.used; ++i) {
    float ms = 0.f;
    HB_CUDA(cudaEventSynchronize(g_prof.b[i]));
    HB_CUDA(cudaEventElapsedTime(&ms, g_prof.a[i], g_prof.b[i]));
    tot += ms;
  }
  *total_ms = tot;
  *n_launches = (int32_t)g_prof.used;
  g_prof.used = 0;
  return HB_OK;
}

int32_t hb_guard_stats(uint64_t *rows_flagged, int32_t reset) {
  if (!rows_flagged) return HB_ERR_INVALID;
  unsigned long long v[2] = {0, 0};
  const int s = guard_stats(v, reset);
  rows_flagged[0] = v[0];
  rows_flagged[1] = v[1];
  return s;
}

int64_t hb_num_params(int64_t d, const hb_model_spec_t *spec) {
  ModelSpec sp;
  if (!build_spec(d, spec, sp)) return -1;
  return sp.P();
}
int64_t hb_fit_workspace_bytes_ex(int64_t n, int64_t d, const hb_model_spec_t *spec) {
  ModelSpec sp;
  if (n <= 0 || !build_spec(d, spec, sp)) return -1;
  return (int64_t)carve_fit(nullptr, n, sp).total;
}
int64_t hb_fit_workspace_bytes(int64_t n, int64_t d) { return d <= 0 ? -1 : hb_fit_workspace_bytes_ex(n, d, nullptr); }
int64_t hb_posterior_workspace_bytes(int64_t n, int64_t d, int64_t m_chunk) {
  if (n <= 0 || d < 0 || m_chunk <= 0) return -1;
  return (int64_t)posterior_ws_bytes(round_up(n, TILE), d, m_chunk);
}
int64_t hb_pareto_workspace_bytes(int64_t m) {
  if (m <= 0) return -1;
  return (int64_t)pareto_ws_bytes(m);
}

int32_t hb_transform_hypers(const float *raw, int64_t d, float noise_lb, float *hyp, void *stream) {
  ModelSpec sp;
  if (!raw || !hyp || d <= 0 || !build_spec(d, nullptr, sp)) return HB_ERR_INVALID;
  return launch_transform_hypers(raw, sp, noise_lb, hyp, (cudaStream_t)stream);
}

int32_t hb_median_pdist(const float *Xt, int64_t n, int64_t d, const int32_t *idx, int64_t k, float clamp_min,
                        float *out, void *stream) {
  if (!Xt || !out || n <= 0) return HB_ERR_INVALID;
  return launch_median_pdist(Xt, round_up(n, TILE), d, idx, k, clamp_min, out, (cudaStream_t)stream);
}

int32_t hb_gram(const float *Xt, int64_t n, int64_t d, const float *hyp, int32_t kern, const float *noise_diag,
                float jitter, float *K, void *stream) {
  ModelSpec sp;
  if (!Xt || !hyp || !K || d <= 0 || !build_spec(d, nullptr, sp)) return HB_ERR_INVALID;
  return launch_gram(Xt, nullptr, n, round_up(n, TILE), sp, hyp, kern, noise_diag, jitter, K, (cudaStream_t)stream);
}

int32_t hb_cholesky(float *A, int64_t np, float *ws, int32_t *info, void *stream) {
  if (!A || !ws || !info) return HB_ERR_INVALID;
  return launch_cholesky(A, np, ws, info, (cudaStream_t)stream);
}

int32_t hb_tri_inverse(const float *L, int64_t np, float *Linv, float *tmp, void *stream) {
  if (!L || !Linv || !tmp) return HB_ERR_INVALID;
  return launch_tri_inverse(L, np, Linv, tmp, (cudaStream_t)stream);
}

int32_t hb_kinv(const float *Linv, int64_t np, float *Kinv, void *stream) {
  if (!Linv || !Kinv) return HB_ERR_INVALID;
  return launch_kinv(Linv, np, Kinv, (cudaStream_t)stream);
}

int32_t hb_solve_logdet(const float *L, const float *Linv, const float *y, int64_t n, int64_t np, const float *hyp,
                        float *alpha, double *scal, void *ws, void *stream) {
  if (!L || !Linv || !y || !hyp || !alpha || !scal || !ws) return HB_ERR_INVALID;
  return launch_solve_logdet(L, Linv, y, n, np, hyp, alpha, scal, ws, (cudaStream_t)stream);
}

int32_t hb_mll_grad(const float *Xt, int64_t n, int64_t d, const float *raw, const float *hyp, int32_t kern,
                    const float *Kinv, const float *alpha, const double *scal, float noise_guess, float *grad,
                    float *loss, void *ws, void *stream) {
  ModelSpec sp;
  if (!Xt || !raw || !hyp || !Kinv || !alpha || !scal || !grad || !loss || !ws || d <= 0 || !build_spec(d, nullptr, sp))
    return HB_ERR_INVALID;
  return launch_mll_grad(Xt, nullptr, n, round_up(n, TILE), sp, raw, hyp, kern, Kinv, alpha, scal, noise_guess, grad, loss, ws,
                         (cudaStream_t)stream);
}

int32_t hb_psgld_step(float *raw, const float *grad, float *square_avg, int64_t p, float lr, float rms_alpha,
                      float rms_eps, float factor, const float *xi, void *stream) {
  if (!raw || !grad || !square_avg) return HB_ERR_INVALID;
  return launch_psgld(raw, grad, square_avg, p, lr, rms_alpha, rms_eps, factor, xi, (cudaStream_t)stream);
}

int32_t hb_fit_state_ex(void *ws, int64_t n, int64_t d, const hb_model_spec_t *spec, hb_fit_state_t *out) {
  ModelSpec sp;
  if (!ws || !out || n <= 0 || !build_spec(d, spec, sp)) return HB_ERR_INVALID;
  FitWs w = carve_fit(ws, n, sp);
  out->hyp = w.hyp;
  out->L = w.L;
  out->Linv = w.Linv;
  out->alpha = w.alpha;
  out->Zt = w.Zt;
  out->scal = w.scal;
  out->Linv_hi = w.Linv_hi;
  out->Linv_lo = w.Linv_lo;
  out->tab_s = w.tab_s;
  out->emb_meta = w.meta;
  out->grad = w.grad;
  out->loss = w.loss;
  return HB_OK;
}
int32_t hb_fit_state(void *ws, int64_t n, int64_t d, hb_fit_state_t *out) {
  return d <= 0 ? HB_ERR_INVALID : hb_fit_state_ex(ws, n, d, nullptr, out);
}

// uploads the categorical layout arrays + training categories into the workspace and binds the device pointers
static int bind_spec_ws(const hb_model_spec_t *spec, ModelSpec &sp, FitWs &w, const int32_t *Xe, int64_t n, cudaStream_t st) {
  if (sp.e <= 0) return HB_OK;
  if (!Xe) return HB_ERR_INVALID;
  std::vector<int32_t> m;
  fill_meta_host(spec, sp, m);
  HB_CUDA(cudaMemcpyAsync(w.meta, m.data(), m.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  HB_CUDA(cudaStreamSynchronize(st));   // `m` is pageable host memory and dies with this frame
  if (Xe != w.Xe) HB_CUDA(cudaMemcpyAsync(w.Xe, Xe, (size_t)n * sp.e * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
  bind_meta(sp, w.meta, w.Xe);
  return HB_OK;
}

int32_t hb_factorize_ex(const float *Xt, const int32_t *Xe, const float *y, int64_t n, int64_t d, const hb_model_spec_t *spec,
                        const float *raw, int32_t kern, const float *noise_diag, float noise_lb, float *jitter_used, void *ws,
                        int64_t ws_bytes, void *stream) {
  ModelSpec sp;
  if (!y || !raw || !ws || n <= 0 || kern < 0 || kern > 2 || !build_spec(d, spec, sp) || (sp.d > 0 && !Xt)) return HB_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  FitWs w = carve_fit(ws, n, sp);
  if ((size_t)ws_bytes < w.total) return HB_ERR_INVALID;
  const int64_t np = round_up(n, TILE);
  HostStatus *hs = pinned_status();
  if (!hs) return HB_ERR_CUDA;
  int s = bind_spec_ws(spec, sp, w, Xe, n, st);
  if (s != HB_OK) return s;
  s = launch_transform_hypers(raw, sp, noise_lb, w.hyp, st);
  if (s != HB_OK) return s;
  float jitter = 0.0f;
  for (;;) {   // gp.py:140-157 jitter escalation of predict()
    // the prediction state is built ONCE per fit: keep it on the FP32 SIMT pipe (round-to-nearest accumulation);
    // the 3xTF32 tensor path (TMEM accumulation is not RN, ~5e-6 relative) is used for the 100 gradient epochs only
    s = factor_once(Xt, n, np, sp, raw, kern, noise_diag, jitter, w, st, /*allow_tc=*/false);
    if (s != HB_OK) return s;
    HB_CUDA(cudaMemcpyAsync(&hs->info, w.info, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    HB_CUDA(cudaStreamSynchronize(st));
    if (hs->info == 0) break;
    jitter = next_jitter(jitter);
    if (jitter > JITTER_MAX) {
      if (jitter_used) *jitter_used = jitter;
      return HB_ERR_NOT_PD;
    }
  }
  if (jitter_used) *jitter_used = jitter;
  s = launch_tri_inverse(w.L, np, w.Linv, w.tmp, st);
  if (s != HB_OK) return s;
  s = launch_linv_refine(w.L, w.Linv, np, w.tmp, w.tc.T_hi, st);   // Newton step, fp64 residual (scratch: tmp, T_hi)
  if (s != HB_OK) return s;
  // operands of the posterior's tensor-core contraction: two-level fp16 split (h0 in the Linv_hi buffer, h1 in the first
  // half of the Linv_lo buffer, the power-of-two scale right after it)
  s = launch_split_h16(w.Linv, np * np, reinterpret_cast<__half *>(w.Linv_hi), reinterpret_cast<__half *>(w.Linv_lo),
                       w.Linv_lo + np * np / 2, st);
  if (s != HB_OK) return s;
  s = launch_solve_logdet(w.L, w.Linv, y, n, np, w.hyp, w.alpha, w.scal, w.solvews, st);
  if (s != HB_OK) return s;
  return launch_scale_zt(Xt, np, sp, w.hyp, w.Zt, w.dZa, w.dZb, st);   // (embedding rows of Zt: filled by factor_once's gather)
}
int32_t hb_factorize(const float *Xt, const float *y, int64_t n, int64_t d, const float *raw, int32_t kern,
                     const float *noise_diag, float noise_lb, float *jitter_used, void *ws, int64_t ws_bytes,
                     void *stream) {
  if (d <= 0) return HB_ERR_INVALID;
  return hb_factorize_ex(Xt, nullptr, y, n, d, nullptr, raw, kern, noise_diag, noise_lb, jitter_used, ws, ws_bytes, stream);
}

// one MLL forward + backward at `raw` (SURVEY 8b `hb_mll_fwd_bwd`): transform -> [gather] -> Gram -> Cholesky -> L^-1 ->
// alpha / log-det -> K^-1 -> gradient; FP32 SIMT GEMM stages.  Results stay on the device (fit-state grad / loss, `info`).
int32_t hb_mll_fwd_bwd(const float *Xt, const int32_t *Xe, const float *y, int64_t n, int64_t d, const hb_model_spec_t *spec,
                       const float *raw, int32_t kern, const float *noise_diag, float noise_lb, float noise_guess, float jitter,
                       float *grad, float *loss, int32_t *info, void *ws, int64_t ws_bytes, void *stream) {
  ModelSpec sp;
  if (!y || !raw || !ws || !grad || !loss || !info || n <= 0 || kern < 0 || kern > 2 || !build_spec(d, spec, sp) ||
      (sp.d > 0 && !Xt))
    return HB_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  FitWs w = carve_fit(ws, n, sp);
  if ((size_t)ws_bytes < w.total) return HB_ERR_INVALID;
  const int64_t np = round_up(n, TILE);
  int s = bind_spec_ws(spec, sp, w, Xe, n, st);
  if (s != HB_OK) return s;
  s = launch_transform_hypers(raw, sp, noise_lb, w.hyp, st);
  if (s != HB_OK) return s;
  s = factor_once(Xt, n, np, sp, raw, kern, noise_diag, jitter, w, st, /*allow_tc=*/false);
  if (s != HB_OK) return s;
  s = launch_tri_inverse(w.L, np, w.Linv, w.tmp, st);
  if (s != HB_OK) return s;
  s = launch_solve_logdet(w.L, w.Linv, y, n, np, w.hyp, w.alpha, w.scal, w.solvews, st);
  if (s != HB_OK) return s;
  s = launch_kinv(w.Linv, np, w.tmp, st);
  if (s != HB_OK) return s;
  s = launch_mll_grad(sp.warp ? w.Zt : Xt, w.Ets, n, np, sp, raw, w.hyp, kern, w.tmp, w.alpha, w.scal, noise_guess, w.grad, w.loss,
                      w.gradws, st, w.dZa, w.dZb);
  if (s != HB_OK) return s;
  HB_CUDA(cudaMemcpyAsync(grad, w.grad, sp.P() * sizeof(float), cudaMemcpyDeviceToDevice, st));
  HB_CUDA(cudaMemcpyAsync(loss, w.loss, sizeof(float), cudaMemcpyDeviceToDevice, st));
  HB_CUDA(cudaMemcpyAsync(info, w.info, sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
  return HB_OK;
}

int32_t hb_fit_ex(const float *Xt, const int32_t *Xe, const float *y, int64_t n, int64_t d, const hb_model_spec_t *spec,
                  float *raw, int32_t kern, const float *noise_diag, float noise_lb, float noise_guess, float lr,
                  int32_t num_epochs, const float *langevin, float *losses, void *ws, int64_t ws_bytes, void *stream) {
  ModelSpec sp;
  if (!y || !raw || !ws || n <= 0 || kern < 0 || kern > 2 || num_epochs < 0 || !build_spec(d, spec, sp) || (sp.d > 0 && !Xt))
    return HB_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  FitWs w = carve_fit(ws, n, sp);
  if ((size_t)ws_bytes < w.total) return HB_ERR_INVALID;
  const int64_t np = round_up(n, TILE);
  const int64_t P = sp.P();
  HostStatus *hs = pinned_status();
  if (!hs) return HB_ERR_CUDA;
  {
    const int s = bind_spec_ws(spec, sp, w, Xe, n, st);
    if (s != HB_OK) return s;
  }
  HB_CUDA(cudaMemsetAsync(w.sq, 0, P * sizeof(float), st));
  HB_CUDA(cudaMemsetAsync(w.info, 0, 4 * sizeof(int32_t), st));   // status, epoch counter, replay slot
  bool zeroed = false;                           // triangular complements of Linv / U zero-filled once per fit
  const int pretrain = num_epochs / 10;          // gp.py:99 pretrain_step = num_epochs // 10
  const float factor = 1.0f / (float)n;          // gp.py:99 factor = 1 / y.shape[0]

  // one epoch = transform -> [gather] -> Gram -> Cholesky -> L^-1 -> alpha / log-det -> K^-1 -> gradient -> guarded pSGLD step
  auto enqueue_epoch = [&](float jitter, cudaStream_t s_) -> int {
    int s = launch_transform_hypers(raw, sp, noise_lb, w.hyp, s_);
    if (s != HB_OK) return s;
    s = factor_once(Xt, n, np, sp, raw, kern, noise_diag, jitter, w, s_);
    if (s != HB_OK) return s;
    if (fit_use_tc()) {
      s = launch_tri_inverse_tc(w.L, np, w.Linv, w.tc, !zeroed, s_);
      zeroed = true;
    } else {
      s = launch_tri_inverse(w.L, np, w.Linv, w.tmp, s_);
    }
    if (s != HB_OK) return s;
    s = launch_solve_logdet(w.L, w.Linv, y, n, np, w.hyp, w.alpha, w.scal, w.solvews, s_);
    if (s != HB_OK) return s;
    s = fit_use_tc() ? launch_kinv_tc(np, w.tmp, w.tc, s_) : launch_kinv(w.Linv, np, w.tmp, s_);
    if (s != HB_OK) return s;
    s = launch_mll_grad(sp.warp ? w.Zt : Xt, w.Ets, n, np, sp, raw, w.hyp, kern, w.tmp, w.alpha, w.scal, noise_guess, w.grad, w.loss,
                        w.gradws, s_, w.dZa, w.dZb);
    if (s != HB_OK) return s;
    psgld_guarded_kernel<<<1, 256, 0, s_>>>(raw, w.grad, w.sq, (int)P, lr, 0.99f, 1e-8f, factor, langevin, pretrain, w.info,
                                           w.loss, w.status, w.hyp, sp.H(), sp.warp == 2 ? sp.i_wa() : 0,
                                           sp.warp == 2 ? sp.i_wa() + sp.n_w() : 0);
    count_launches(1);
    HB_LAUNCH_CHECK("psgld_guarded");
    return HB_OK;
  };
  // epoch `ep` with the jitter ladder of gp.py:104-126, one host synchronisation per attempt
  bool hopeless = false;
  int hopeless_from = 0;
  auto slow_epoch = [&](int ep) -> int {
    float jitter = 0.0f;
    for (;;) {
      HB_CUDA(cudaMemsetAsync(w.info + 2, 0, sizeof(int32_t), st));           // replay slot 0
      const int s = enqueue_epoch(jitter, st);
      if (s != HB_OK) return s;
      HB_CUDA(cudaMemcpyAsync(hs->batch, w.status, 2 * sizeof(float), cudaMemcpyDeviceToHost, st));
      HB_CUDA(cudaStreamSynchronize(st));
      int32_t info;
      memcpy(&info, &hs->batch[0], sizeof(info));
      if (info == 0) {
        if (losses) losses[ep] = hs->batch[1];
        return HB_OK;
      }
      if (info == -1) {            // hopeless (see psgld_guarded_kernel): this and every later epoch is given up
        hopeless = true;
        hopeless_from = ep;
        return HB_OK;
      }
      jitter = next_jitter(jitter);
      if (jitter > JITTER_MAX) {   // "jitter is too large, give up fitting GP": epoch skipped, gp.py:121-122
        if (losses) losses[ep] = INFINITY;
        hs->set_epoch = ep + 1;     // the device counter only advances on success
        HB_CUDA(cudaMemcpyAsync(w.info + 1, &hs->set_epoch, sizeof(int32_t), cudaMemcpyHostToDevice, st));
        HB_CUDA(cudaStreamSynchronize(st));
        return HB_OK;
      }
    }
  };

  int ep = 0;
  if (num_epochs > 0) {   // first epoch on the plain path: it also builds every lazily created table / attribute
    const int s = slow_epoch(0);
    if (s != HB_OK) return s;
    ep = 1;
  }
  // Remaining epochs: capture ONE epoch (jitter 0) into a CUDA graph and replay it FIT_BATCH times per host
  // synchronisation.  A failed factorisation leaves the hypers, the RMS state and the device epoch counter untouched
  // (the pSGLD kernel is guarded), so every later replay of the batch fails the same way; the host then runs that epoch
  // through the jitter ladder on the plain path and resumes.  HEBO_B200_FIT_GRAPH=0 disables the graph path.
  static const bool graph_on = [] {
    const char *e = getenv("HEBO_B200_FIT_GRAPH"), *t = getenv("HEBO_B200_CHOL_TIMING");
    return !(e && e[0] == '0') && !(t && t[0] == '1');
  }();
  cudaGraphExec_t exec = nullptr;
  long long launches_per_epoch = 0;
  if (graph_on && num_epochs - ep >= 4) {
    static cudaStream_t gs_dev[MAX_DEVICES] = {};   // one capture stream per device
    int cur_dev = 0;
    cudaGetDevice(&cur_dev);
    cudaStream_t &gs = gs_dev[(cur_dev >= 0 && cur_dev < MAX_DEVICES) ? cur_dev : 0];
    if (!gs && cudaStreamCreateWithFlags(&gs, cudaStreamNonBlocking) != cudaSuccess) gs = nullptr;
    if (gs) {
      HB_CUDA(cudaStreamSynchronize(st));
      cudaGraph_t graph = nullptr;
      const long long before = g_launches.load();
      if (cudaStreamBeginCapture(gs, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
        const int s = enqueue_epoch(0.0f, gs);
        const cudaError_t e = cudaStreamEndCapture(gs, &graph);
        if (s == HB_OK && e == cudaSuccess && graph && cudaGraphInstantiate(&exec, graph, 0) == cudaSuccess) {
          launches_per_epoch = g_launches.load() - before;
        } else {
          exec = nullptr;
        }
        if (graph) cudaGraphDestroy(graph);
      }
      g_launches = before;       // nothing was launched by the capture itself
      (void)cudaGetLastError();  // a failed capture must not poison the plain path
    }
  }
  int batch = FIT_BATCH;
  while (ep < num_epochs) {
    if (hopeless) break;
    if (!exec) {
      const int s = slow_epoch(ep);
      if (s != HB_OK) return s;
      ++ep;
      continue;
    }
    int B = batch < FIT_BATCH ? batch : FIT_BATCH;   // ramps 1, 2, 4, .. after a failure: a failing epoch wastes the rest
    if (B > num_epochs - ep) B = num_epochs - ep;    // of its batch, and failures come in runs (gp.py:117-126 territory)
    HB_CUDA(cudaMemsetAsync(w.info + 2, 0, sizeof(int32_t), st));
    for (int b = 0; b < B; ++b) HB_CUDA(cudaGraphLaunch(exec, st));
    count_launches(launches_per_epoch * B);
    HB_CUDA(cudaMemcpyAsync(hs->batch, w.status, (size_t)B * 2 * sizeof(float), cudaMemcpyDeviceToHost, st));
    HB_CUDA(cudaStreamSynchronize(st));
    int done = 0;
    for (; done < B; ++done) {
      int32_t info;
      memcpy(&info, &hs->batch[2 * done], sizeof(info));
      if (info != 0) break;
      if (losses) losses[ep + done] = hs->batch[2 * done + 1];
    }
    ep += done;
    batch = (done < B) ? 1 : (2 * batch > FIT_BATCH ? FIT_BATCH : 2 * batch);
    if (done < B) {   // epoch `ep` needs jitter: plain path with the ladder, then back to the graph
      const int s = slow_epoch(ep);
      if (s != HB_OK) {
        cudaGraphExecDestroy(exec);
        return s;
      }
      ++ep;
    }
  }
  if (exec) cudaGraphExecDestroy(exec);
  if (hopeless && losses)          // "jitter is too large, give up fitting GP" for that and every remaining epoch
    for (int e = hopeless_from; e < num_epochs; ++e) losses[e] = INFINITY;
  return hb_factorize_ex(Xt, w.Xe, y, n, d, spec, raw, kern, noise_diag, noise_lb, nullptr, ws, ws_bytes, stream);
}
int32_t hb_fit(const float *Xt, const float *y, int64_t n, int64_t d, float *raw, int32_t kern,
               const float *noise_diag, float noise_lb, float noise_guess, float lr, int32_t num_epochs,
               const float *langevin, float *losses, void *ws, int64_t ws_bytes, void *stream) {
  if (d <= 0) return HB_ERR_INVALID;
  return hb_fit_ex(Xt, nullptr, y, n, d, nullptr, raw, kern, noise_diag, noise_lb, noise_guess, lr, num_epochs, langevin, losses,
                   ws, ws_bytes, stream);
}

int32_t hb_posterior_mace_ex(const float *Xs, const int32_t *Xe_s, int64_t m, int64_t rng_offset, int64_t n, int64_t d,
                             const hb_model_spec_t *spec,
                             const int32_t *emb_meta, const float *tab_s, const float *x_mul, const float *x_add,
                             const float *Zt, const float *alpha, const float *Linv, const float *Linv_hi,
                             const float *Linv_lo, const float *hyp, int32_t kern, float y_mean, float y_std, int32_t pred_likeli,
                             float tau, float kappa, float eps, const float *xi1, const float *xi2, uint64_t seed, float *F,
                             float *mu, float *var, void *ws, int64_t ws_bytes, int64_t m_chunk, void *stream) {
  ModelSpec sp;
  if (!build_spec(d, spec, sp)) return HB_ERR_INVALID;
  if ((sp.d > 0 && (!Xs || !x_mul || !x_add)) || !Zt || !alpha || !Linv || !hyp || !ws) return HB_ERR_INVALID;
  if (sp.e > 0 && (!Xe_s || !emb_meta || !tab_s)) return HB_ERR_INVALID;
  if (!F && !mu && !var) return HB_ERR_INVALID;
  if ((Linv_hi == nullptr) != (Linv_lo == nullptr)) return HB_ERR_INVALID;
  bind_meta(sp, emb_meta, nullptr);
  return launch_posterior_mace(Xs, Xe_s, m, rng_offset, n, round_up(n, TILE), sp, tab_s, x_mul, x_add, Zt, alpha, Linv, Linv_hi, Linv_lo, hyp,
                               kern, y_mean, y_std, pred_likeli, tau, kappa, eps, xi1, xi2, seed, F, mu, var, ws, ws_bytes,
                               m_chunk, (cudaStream_t)stream);
}
int32_t hb_posterior_mace(const float *Xs, int64_t m, int64_t n, int64_t d, const float *x_mul, const float *x_add,
                          const float *Zt, const float *alpha, const float *Linv, const float *Linv_hi,
                          const float *Linv_lo, const float *hyp, int32_t kern, float y_mean, float y_std, int32_t pred_likeli, float tau, float kappa, float eps,
                          const float *xi1, const float *xi2, uint64_t seed, float *F, float *mu, float *var,
                          void *ws, int64_t ws_bytes, int64_t m_chunk, void *stream) {
  if (d <= 0) return HB_ERR_INVALID;
  return hb_posterior_mace_ex(Xs, nullptr, m, 0, n, d, nullptr, nullptr, nullptr, x_mul, x_add, Zt, alpha, Linv, Linv_hi, Linv_lo, hyp,
                              kern, y_mean, y_std, pred_likeli, tau, kappa, eps, xi1, xi2, seed, F, mu, var, ws, ws_bytes, m_chunk,
                              stream);
}

int32_t hb_posterior_grad_ex(const float *Xs, const int32_t *Xe_s, int64_t m, int64_t n, int64_t d, const hb_model_spec_t *spec,
                             const int32_t *emb_meta, const float *tab_s, const float *x_mul, const float *x_add,
                             const float *Zt, const float *alpha, const float *Linv, const float *hyp, int32_t kern, float y_mean,
                             float y_std, int32_t pred_likeli, float *mu, float *var, float *dmu, float *dvar, void *ws,
                             int64_t ws_bytes, int64_t m_chunk, void *stream) {
  ModelSpec sp;
  if (d <= 0 || !build_spec(d, spec, sp)) return HB_ERR_INVALID;
  if (!Xs || !x_mul || !x_add || !Zt || !alpha || !Linv || !hyp || !ws || !mu || !var || !dmu || !dvar) return HB_ERR_INVALID;
  if (sp.e > 0 && (!Xe_s || !emb_meta || !tab_s)) return HB_ERR_INVALID;
  bind_meta(sp, emb_meta, nullptr);
  return launch_posterior_grad(Xs, Xe_s, m, n, round_up(n, TILE), sp, tab_s, x_mul, x_add, Zt, alpha, Linv, hyp, kern, y_mean, y_std,
                               pred_likeli, mu, var, dmu, dvar, ws, ws_bytes, m_chunk, (cudaStream_t)stream);
}
int32_t hb_posterior_grad(const float *Xs, int64_t m, int64_t n, int64_t d, const float *x_mul, const float *x_add,
                          const float *Zt, const float *alpha, const float *Linv, const float *hyp, int32_t kern, float y_mean,
                          float y_std, int32_t pred_likeli, float *mu, float *var, float *dmu, float *dvar, void *ws,
                          int64_t ws_bytes, int64_t m_chunk, void *stream) {
  return hb_posterior_grad_ex(Xs, nullptr, m, n, d, nullptr, nullptr, nullptr, x_mul, x_add, Zt, alpha, Linv, hyp, kern, y_mean, y_std,
                              pred_likeli, mu, var, dmu, dvar, ws, ws_bytes, m_chunk, stream);
}

int64_t hb_sample_workspace_bytes(int64_t n, int64_t d, const hb_model_spec_t *spec, int64_t m) {
  ModelSpec sp;
  if (n <= 0 || m <= 0 || !build_spec(d, spec, sp)) return -1;
  return (int64_t)sample_ws_bytes(round_up(n, TILE), sp.dtot(), m);
}

int32_t hb_sample_y(const float *Xs, const int32_t *Xe_s, int64_t m, int64_t n, int64_t d, const hb_model_spec_t *spec,
                    const int32_t *emb_meta, const float *tab_s, const float *x_mul, const float *x_add, const float *Zt,
                    const float *alpha, const float *Linv, const float *hyp, const float *hyp_host, int32_t kern, float y_mean,
                    float y_std, int32_t pred_likeli, const float *z, int32_t n_samples, float *out, float *jitter_used, void *ws,
                    int64_t ws_bytes, void *stream) {
  ModelSpec sp;
  if (!build_spec(d, spec, sp)) return HB_ERR_INVALID;
  if ((sp.d > 0 && (!Xs || !x_mul || !x_add)) || !Zt || !alpha || !Linv || !hyp || !hyp_host || !z || !out || !ws) return HB_ERR_INVALID;
  if (sp.e > 0 && (!Xe_s || !emb_meta || !tab_s)) return HB_ERR_INVALID;
  bind_meta(sp, emb_meta, nullptr);
  return launch_sample_y(Xs, Xe_s, m, n, round_up(n, TILE), sp, tab_s, x_mul, x_add, Zt, alpha, Linv, hyp, hyp_host, kern, y_mean,
                         y_std, pred_likeli, z, n_samples, out, jitter_used, ws, ws_bytes, (cudaStream_t)stream);
}

int32_t hb_mace_epilogue(const float *mu, const float *var, int64_t m, float noise_var, float tau, float kappa,
                         float eps, const float *xi1, const float *xi2, uint64_t seed, float *F, void *stream) {
  if (!mu || !var || !F) return HB_ERR_INVALID;
  return launch_mace_only(mu, var, m, noise_var, tau, kappa, eps, xi1, xi2, seed, F, (cudaStream_t)stream);
}

int32_t hb_general_acq_epilogue(const float *mu, const float *var, int64_t m, int32_t num_obj, int32_t num_constr,
                                const float *noise_var, float kappa, float c_kappa, int32_t use_noise, const float *xi, uint64_t seed,
                                int64_t rng_offset, float *out, float *cv, void *stream) {
  if (!mu || !var || !out || (use_noise && !noise_var)) return HB_ERR_INVALID;
  return launch_general_acq(mu, var, m, num_obj, num_constr, noise_var, kappa, c_kappa, use_noise, xi, seed, rng_offset, out, cv,
                            (cudaStream_t)stream);
}

int32_t hb_pareto_front(const float *F, int64_t m, int32_t K, int64_t ldf, const float *cv, int32_t *idx_out, int32_t *count,
                        void *ws, int64_t ws_bytes, void *stream) {
  if (!F || !idx_out || !count || !ws || K < 1 || K > 8 || ldf < K) return HB_ERR_INVALID;
  return launch_pareto(F, m, K, ldf, cv, idx_out, count, ws, ws_bytes, (cudaStream_t)stream);
}

int32_t hb_pareto_front3(const float *F, int64_t m, int32_t *idx_out, int32_t *count, void *ws, int64_t ws_bytes,
                         void *stream) {
  if (!F || !idx_out || !count || !ws) return HB_ERR_INVALID;
  return launch_pareto3(F, m, idx_out, count, ws, ws_bytes, (cudaStream_t)stream);
}

int64_t hb_front_merge_workspace_bytes(int64_t world, int64_t capacity) {
  if (world <= 0 || capacity <= 0) return -1;
  return (int64_t)front_merge_ws_bytes(world, capacity);
}

int32_t hb_front_pack(const float *F, const float *mu, const float *var, const int32_t *idx, const int32_t *count,
                      int64_t row_offset, int64_t capacity, float *out, void *stream) {
  if (!F || !idx || !count || !out) return HB_ERR_INVALID;
  return launch_front_pack(F, mu, var, idx, count, row_offset, capacity, out, (cudaStream_t)stream);
}

int32_t hb_front_merge(const float *all_buf, int64_t world, int64_t capacity, float *out, void *ws, int64_t ws_bytes,
                       void *stream) {
  if (!all_buf || !out || !ws) return HB_ERR_INVALID;
  return launch_front_merge(all_buf, world, capacity, out, ws, ws_bytes, (cudaStream_t)stream);
}

int32_t hb_nsga2_init(float *X, int64_t pop, int64_t D, int64_t d, const int32_t *kind, const float *lb, const float *ub,
                      const float *fixed, const float *init, int64_t n_init, uint64_t seed, float *Xc, int32_t *Xe, void *stream) {
  if (!X || !kind || !lb || !ub || !fixed || (n_init > 0 && !init) || (d > 0 && !Xc) || (D > d && !Xe)) return HB_ERR_INVALID;
  return launch_nsga_init(X, pop, D, d, kind, lb, ub, fixed, init, n_init, seed, Xc, Xe, (cudaStream_t)stream);
}

int32_t hb_nsga2_mate(const float *X, int64_t pop, int64_t D, int64_t d, const int32_t *kind, const float *lb, const float *ub,
                      const float *fixed, uint64_t seed, int32_t generation, float *C, float *Cc, int32_t *Ce, void *stream) {
  if (!X || !kind || !lb || !ub || !fixed || !C || (d > 0 && !Cc) || (D > d && !Ce)) return HB_ERR_INVALID;
  return launch_nsga_mate(X, pop, D, d, kind, lb, ub, fixed, seed, generation, C, Cc, Ce, (cudaStream_t)stream);
}

int32_t hb_nsga2_survive(const float *X, const float *F, const float *C, const float *FC, int64_t pop, int64_t D, int64_t d,
                         float *X_next, float *F_next, float *Xc_next, int32_t *Xe_next, void *stream) {
  if (!X || !F || !C || !FC || !X_next || !F_next || (d > 0 && !Xc_next) || (D > d && !Xe_next)) return HB_ERR_INVALID;
  return launch_nsga_survive(X, F, C, FC, pop, D, d, X_next, F_next, Xc_next, Xe_next, (cudaStream_t)stream);
}

int32_t hb_nsga2_survive_k(const float *X, const float *F, const float *CV, const float *C, const float *FC, const float *CVC,
                           int64_t pop, int64_t D, int64_t d, int32_t K, float *X_next, float *F_next, float *CV_next,
                           float *Xc_next, int32_t *Xe_next, void *stream) {
  if (!X || !F || !C || !FC || !X_next || !F_next || (d > 0 && !Xc_next) || (D > d && !Xe_next)) return HB_ERR_INVALID;
  if (K < 1 || K > 8 || (CV == nullptr) != (CVC == nullptr) || (CV && !CV_next)) return HB_ERR_INVALID;
  return launch_nsga_survive_k(X, F, CV, C, FC, CVC, pop, D, d, K, X_next, F_next, CV_next, Xc_next, Xe_next, (cudaStream_t)stream);
}

}  // extern "C"
