// Device-resident NSGA-II for the acquisition optimiser (SURVEY 8f-1): the role pymoo's NSGA2 + MixedVariableMating play in
// HEBO/hebo/acq_optimizers/evolution_optimizer.py:107-160 (pop 100, `iters` generations, Real -> SBX + polynomial
// mutation, Integer -> the same + rounding repair, Choice -> uniform crossover + random-resample mutation, duplicate
// elimination, rank-and-crowding survival; variable typing as evolution_optimizer.py:26-41).  pymoo is a third-party
// dependency that is not installed here: the operators follow the published algorithms (Deb et al. 2002; Deb & Agrawal
// SBX eta = 15, pair probability 0.9, per-variable 0.5; Deb & Goyal PM eta = 20, per-variable min(0.5, 1/D)) -- pymoo's
// random stream is not reproduced.  The population never leaves the device: one generation = mate (1 launch) -> fused
// posterior + MACE on the offspring (the C-ABI call the Sobol path uses) -> survive (1 launch), no host synchronisation.
//
// Layout: X [P, D] fp32 in the optimisation space (numeric columns first, then the categorical indices as floats);
// kind[D]: 0 real, 1 integer, 2 choice; lb / ub [D]; fixed[D] (NaN = free, else the value of a `fix_input` column).
#include "kernels.h"

namespace hb {

__device__ __forceinline__ void philox4(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint64_t seed, float (&u)[4]) {
  uint32_t c[4] = {c0, c1, c2, c3};
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(M0, c[0]), lo0 = M0 * c[0];
    const uint32_t hi1 = __umulhi(M1, c[2]), lo1 = M1 * c[2];
    const uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
    c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) u[i] = ((float)c[i] + 0.5f) * 2.3283064365386963e-10f;   // (0, 1)
}

__device__ __forceinline__ float repair(float v, int kind, float lo, float hi, float fixed) {
  if (!isnan(fixed)) return fixed;
  if (kind != 0) v = rintf(v);
  return fminf(fmaxf(v, lo), hi);
}

// split a float row of the optimisation space into the model's inputs: Xc [d] fp32, Xe [e] int32
__device__ __forceinline__ void split_row(const float *row, int d, int e, float *xc, int32_t *xe) {
  for (int k = 0; k < d; ++k) xc[k] = row[k];
  for (int k = 0; k < e; ++k) xe[k] = (int32_t)rintf(row[d + k]);
}

// initial population: uniform in the box (evolution_optimizer.py:44-55 with the default sobol_init flag samples
// uniformly), typed repair, row 0.. = the initial suggestions (prepended, :56-57)
__global__ void nsga_init_kernel(float *__restrict__ X, int P, int D, int d, const int32_t *__restrict__ kind,
                                 const float *__restrict__ lb, const float *__restrict__ ub, const float *__restrict__ fixed,
                                 const float *__restrict__ init, int n_init, uint64_t seed, float *__restrict__ Xc,
                                 int32_t *__restrict__ Xe) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  float *row = X + (int64_t)p * D;
  for (int k = 0; k < D; k += 4) {
    float u[4];
    philox4((uint32_t)p, 0xFFFFFFFFu, (uint32_t)k, 1u, seed, u);
    for (int j = 0; j < 4 && k + j < D; ++j) {
      const int c = k + j;
      float v = (p < n_init) ? init[(int64_t)p * D + c] : lb[c] + (ub[c] - lb[c]) * u[j];
      if (kind[c] == 2 && p >= n_init) v = floorf(lb[c] + (ub[c] - lb[c] + 1.0f) * u[j]);   // categories equally likely
      row[c] = repair(v, kind[c], lb[c], ub[c], fixed[c]);
    }
  }
  split_row(row, d, D - d, Xc + (int64_t)p * d, Xe + (int64_t)p * (D - d));
}

// one thread per mating: two random parents -> two children (rows 2t, 2t + 1 of the offspring buffers)
__global__ void nsga_mate_kernel(const float *__restrict__ X, int P, int D, int d, const int32_t *__restrict__ kind,
                                 const float *__restrict__ lb, const float *__restrict__ ub, const float *__restrict__ fixed,
                                 uint64_t seed, int gen, float pm_prob, float *__restrict__ C, float *__restrict__ Cc,
                                 int32_t *__restrict__ Ce) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (2 * t >= P) return;
  const float sbx_eta = 15.0f, sbx_prob = 0.9f, sbx_var = 0.5f, pm_eta = 20.0f;
  float u[4];
  philox4((uint32_t)t, (uint32_t)gen, 0xFFFFFFF0u, 2u, seed, u);
  const int pa = min((int)(u[0] * P), P - 1), pb = min((int)(u[1] * P), P - 1);
  const bool do_pair = u[2] < sbx_prob;
  const float *A = X + (int64_t)pa * D, *B = X + (int64_t)pb * D;
  float *c1 = C + (int64_t)(2 * t) * D, *c2 = C + (int64_t)min(2 * t + 1, P - 1) * D;
  const bool second = 2 * t + 1 < P;
  for (int k = 0; k < D; ++k) {
    float v[4], w[4];
    philox4((uint32_t)t, (uint32_t)gen, (uint32_t)k, 3u, seed, v);
    philox4((uint32_t)t, (uint32_t)gen, (uint32_t)k, 4u, seed, w);
    const float lo = lb[k], hi = ub[k];
    float x1 = A[k], x2 = B[k];
    if (kind[k] == 2) {                                   // Choice: uniform crossover, random-resample mutation
      if (do_pair && v[0] < 0.5f) { const float s = x1; x1 = x2; x2 = s; }
      if (v[1] < pm_prob) x1 = floorf(lo + (hi - lo + 1.0f) * v[2]);
      if (w[1] < pm_prob) x2 = floorf(lo + (hi - lo + 1.0f) * w[2]);
    } else {
      // ---- SBX with bounds
      const float y1 = fminf(x1, x2), y2 = fmaxf(x1, x2), diff = y2 - y1;
      if (do_pair && v[0] < sbx_var && diff > 1e-14f) {
        const float uu = v[1], ex = 1.0f / (sbx_eta + 1.0f);
        auto betaq = [&](float beta) {
          const float alpha = 2.0f - powf(beta, -(sbx_eta + 1.0f));
          const float inner = (uu <= 1.0f / alpha) ? uu * alpha : 1.0f / fmaxf(2.0f - uu * alpha, 1e-30f);
          return powf(inner, ex);
        };
        float a = 0.5f * ((y1 + y2) - betaq(1.0f + 2.0f * (y1 - lo) / diff) * diff);
        float b = 0.5f * ((y1 + y2) + betaq(1.0f + 2.0f * (hi - y2) / diff) * diff);
        if (v[2] < 0.5f) { const float s = a; a = b; b = s; }
        x1 = a;
        x2 = b;
      }
      // ---- polynomial mutation
      const float span = hi - lo, mp = 1.0f / (pm_eta + 1.0f);
      auto pm = [&](float x, float um) {
        const float d1 = (x - lo) / span, d2 = (hi - x) / span;
        const float dq = um < 0.5f ? powf(2.0f * um + (1.0f - 2.0f * um) * powf(1.0f - d1, pm_eta + 1.0f), mp) - 1.0f
                                   : 1.0f - powf(2.0f * (1.0f - um) + 2.0f * (um - 0.5f) * powf(1.0f - d2, pm_eta + 1.0f), mp);
        return x + dq * span;
      };
      if (span > 0.0f) {
        x1 = fminf(fmaxf(x1, lo), hi);
        x2 = fminf(fmaxf(x2, lo), hi);
        if (v[3] < pm_prob) x1 = pm(x1, w[0]);
        if (w[3] < pm_prob) x2 = pm(x2, w[1]);
      }
    }
    c1[k] = repair(x1, kind[k], lo, hi, fixed[k]);
    if (second) c2[k] = repair(x2, kind[k], lo, hi, fixed[k]);
  }
  split_row(c1, d, D - d, Cc + (int64_t)(2 * t) * d, Ce + (int64_t)(2 * t) * (D - d));
  if (second) split_row(c2, d, D - d, Cc + (int64_t)(2 * t + 1) * d, Ce + (int64_t)(2 * t + 1) * (D - d));
}

// ---- rank-and-crowding survival of the merged population (pop rows 0..P-1, offspring rows P..2P-1), one CTA, K objectives.
// Without constraints (CV == nullptr) every row takes part; a non-finite objective becomes +inf and a duplicate child
// all +inf, so they only fill slots nothing else can.  With constraints (CV / CVC [P] = sum_j max(0, g_j), pymoo 0.6 calc_cv
// as recalled; evolution_optimizer.py:104-105 hands pymoo F and G) the filter_infeasible rule of pymoo's Survival.do:
// the feasible rows (cv <= 0, finite objectives, not a duplicate) go through rank-and-crowding for min(n_feasible, P) slots,
// the remaining slots go to the other rows in ascending cv (lower merged index first on ties), duplicates and rows with a
// non-finite objective or a NaN cv last.
constexpr int NSGA_MAX = 512;
template <int K>
__global__ void __launch_bounds__(NSGA_MAX) nsga_survive_kernel(const float *__restrict__ X, const float *__restrict__ F,
                                                                const float *__restrict__ CV, const float *__restrict__ C,
                                                                const float *__restrict__ FC, const float *__restrict__ CVC,
                                                                int P, int D, int d, float *__restrict__ Xn,
                                                                float *__restrict__ Fn, float *__restrict__ CVn,
                                                                float *__restrict__ Xcn, int32_t *__restrict__ Xen) {
  __shared__ float f[NSGA_MAX][K];
  __shared__ int ndom[NSGA_MAX], rank[NSGA_MAX], order[NSGA_MAX];
  __shared__ float crowd[NSGA_MAX], cvk[NSGA_MAX];
  __shared__ unsigned char infront[NSGA_MAX], keep[NSGA_MAX], part[NSGA_MAX], bad[NSGA_MAX];
  __shared__ int cnt, cum, r_cut, need, nfeas;
  const int N = 2 * P, i = threadIdx.x;
  const bool on = i < N;
  const bool constrained = CV != nullptr;
  if (i == 0) nfeas = 0;
  if (on) {
    const float *src = i < P ? F + (int64_t)i * K : FC + (int64_t)(i - P) * K;
    bool finite = true;
    for (int k = 0; k < K; ++k) {
      const float v = src[k];
      finite &= isfinite(v);
      f[i][k] = isfinite(v) ? v : INFINITY;                // NaN / inf objectives never survive (evolution_optimizer.py:104 F)
    }
    const float c = constrained ? (i < P ? CV[i] : CVC[i - P]) : 0.0f;
    bad[i] = constrained && (!finite || isnan(c));
    cvk[i] = bad[i] ? 0.0f : c;
    rank[i] = -1;
    keep[i] = 0;
    infront[i] = 0;
  }
  __syncthreads();
  if (on && i >= P) {
    // duplicate elimination (pymoo MixedVariableDuplicateElimination): a child equal to a population member or to an
    // earlier child is discarded
    const float *me = C + (int64_t)(i - P) * D;
    bool dup = false;
    for (int j = 0; j < i && !dup; ++j) {
      const float *o = j < P ? X + (int64_t)j * D : C + (int64_t)(j - P) * D;
      bool same = true;
      for (int k = 0; k < D && same; ++k) same = fabsf(o[k] - me[k]) <= 1e-16f;
      dup = same;
    }
    if (dup) {
      for (int k = 0; k < K; ++k) f[i][k] = INFINITY;
      if (constrained) {
        bad[i] = 1;
        cvk[i] = 0.0f;
      }
    }
  }
  __syncthreads();
  if (on) {
    part[i] = !constrained || (!bad[i] && cvk[i] <= 0.0f);
    if (constrained && part[i]) atomicAdd(&nfeas, 1);
  }
  __syncthreads();
  const int Pf = constrained ? min(nfeas, P) : P;          // slots filled by rank-and-crowding
  auto dominates = [&](int j) {
    bool le = true, lt = false;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      le = le && f[j][k] <= f[i][k];
      lt = lt || f[j][k] < f[i][k];
    }
    return le && lt;
  };
  if (on && part[i]) {
    int c = 0;
    for (int j = 0; j < N; ++j) c += (part[j] && dominates(j)) ? 1 : 0;
    ndom[i] = c;
  }
  if (i == 0) { cum = 0; r_cut = -1; need = 0; }
  __syncthreads();
  // ---- front peeling until Pf survivors are covered
  for (int r = 0; r < N && Pf > 0; ++r) {
    if (i == 0) cnt = 0;
    __syncthreads();
    if (on && part[i] && rank[i] < 0 && ndom[i] == 0) {
      infront[i] = 1;
      atomicAdd(&cnt, 1);
    }
    __syncthreads();
    const int c = cnt;
    if (c == 0) break;
    if (on && infront[i]) rank[i] = r;
    if (i == 0) {
      if (r_cut < 0 && cum + c >= Pf) { r_cut = r; need = Pf - cum; }
      cum += c;
    }
    __syncthreads();
    if (r_cut >= 0) break;
    if (on && part[i] && rank[i] < 0) {
      int sub = 0;
      for (int j = 0; j < N; ++j)
        if (infront[j]) sub += dominates(j) ? 1 : 0;
      ndom[i] -= sub;
    }
    __syncthreads();
    if (on) infront[i] = 0;
    __syncthreads();
  }
  // ---- whole fronts below the cut survive; the cut front is truncated by descending crowding distance
  const int rc = r_cut;
  if (on) {
    keep[i] = (rc >= 0 && rank[i] >= 0 && rank[i] < rc) ? 1 : 0;
    crowd[i] = 0.0f;
  }
  __syncthreads();
  const bool mine = on && rc >= 0 && rank[i] == rc;
  for (int k = 0; k < K; ++k) {
    // position of i inside the cut front along objective k (counting sort, ties by index), then its neighbours
    int pos = 0, m = 0;
    float fmin = INFINITY, fmax = -INFINITY;
    if (mine) {
      for (int j = 0; j < N; ++j)
        if (rank[j] == rc) {
          ++m;
          pos += (f[j][k] < f[i][k] || (f[j][k] == f[i][k] && j < i)) ? 1 : 0;
          fmin = fminf(fmin, f[j][k]);
          fmax = fmaxf(fmax, f[j][k]);
        }
      order[pos] = i;
    }
    __syncthreads();
    if (mine) {
      if (pos == 0 || pos == m - 1) crowd[i] = INFINITY;
      else if (fmax > fmin && isfinite(fmax - fmin)) crowd[i] += (f[order[pos + 1]][k] - f[order[pos - 1]][k]) / (fmax - fmin);
    }
    __syncthreads();
  }
  if (mine) {
    int better = 0;
    for (int j = 0; j < N; ++j)
      if (rank[j] == rc) better += (crowd[j] > crowd[i] || (crowd[j] == crowd[i] && j < i)) ? 1 : 0;
    if (better < need) keep[i] = 1;
  }
  // ---- the remaining P - Pf slots: the other rows by (bad, cv, merged index)
  if (constrained && on && !part[i]) {
    int before = 0;
    for (int j = 0; j < N; ++j)
      if (!part[j])
        before += (bad[j] < bad[i] || (bad[j] == bad[i] && (cvk[j] < cvk[i] || (cvk[j] == cvk[i] && j < i)))) ? 1 : 0;
    if (before < P - Pf) keep[i] = 1;
  }
  __syncthreads();
  // ---- stable compaction into the next population
  if (on && keep[i]) {
    int dst = 0;
    for (int j = 0; j < i; ++j) dst += keep[j];
    const float *src = i < P ? X + (int64_t)i * D : C + (int64_t)(i - P) * D;
    float *row = Xn + (int64_t)dst * D;
    for (int k = 0; k < D; ++k) row[k] = src[k];
    for (int k = 0; k < K; ++k) Fn[(int64_t)dst * K + k] = f[i][k];
    if (constrained) CVn[dst] = i < P ? CV[i] : CVC[i - P];
    split_row(src, d, D - d, Xcn + (int64_t)dst * d, Xen + (int64_t)dst * (D - d));
  }
}

int launch_nsga_init(float *X, int64_t P, int64_t D, int64_t d, const int32_t *kind, const float *lb, const float *ub,
                     const float *fixed, const float *init, int64_t n_init, uint64_t seed, float *Xc, int32_t *Xe, cudaStream_t st) {
  if (P <= 0 || D <= 0 || d < 0 || d > D || n_init < 0 || n_init > P) return HB_ERR_INVALID;
  nsga_init_kernel<<<(int)ceil_div(P, 128), 128, 0, st>>>(X, (int)P, (int)D, (int)d, kind, lb, ub, fixed, init, (int)n_init, seed, Xc, Xe);
  count_launches(1);
  HB_LAUNCH_CHECK("nsga_init");
  return HB_OK;
}

int launch_nsga_mate(const float *X, int64_t P, int64_t D, int64_t d, const int32_t *kind, const float *lb, const float *ub,
                     const float *fixed, uint64_t seed, int gen, float *C, float *Cc, int32_t *Ce, cudaStream_t st) {
  if (P <= 0 || D <= 0 || d < 0 || d > D) return HB_ERR_INVALID;
  const float pm_prob = fminf(0.5f, 1.0f / (float)D);
  nsga_mate_kernel<<<(int)ceil_div((P + 1) / 2, 64), 64, 0, st>>>(X, (int)P, (int)D, (int)d, kind, lb, ub, fixed, seed, gen, pm_prob, C, Cc, Ce);
  count_launches(1);
  HB_LAUNCH_CHECK("nsga_mate");
  return HB_OK;
}

int launch_nsga_survive_k(const float *X, const float *F, const float *CV, const float *C, const float *FC, const float *CVC,
                          int64_t P, int64_t D, int64_t d, int K, float *Xn, float *Fn, float *CVn, float *Xcn, int32_t *Xen,
                          cudaStream_t st) {
  if (P <= 0 || 2 * P > NSGA_MAX || D <= 0 || d < 0 || d > D) return HB_ERR_INVALID;
  if ((CV == nullptr) != (CVC == nullptr) || (CV != nullptr && CVn == nullptr)) return HB_ERR_INVALID;
#define HB_SURV(KK) nsga_survive_kernel<KK><<<1, NSGA_MAX, 0, st>>>(X, F, CV, C, FC, CVC, (int)P, (int)D, (int)d, Xn, Fn, CVn, Xcn, Xen)
  switch (K) {
    case 1: HB_SURV(1); break;
    case 2: HB_SURV(2); break;
    case 3: HB_SURV(3); break;
    case 4: HB_SURV(4); break;
    case 5: HB_SURV(5); break;
    case 6: HB_SURV(6); break;
    case 7: HB_SURV(7); break;
    case 8: HB_SURV(8); break;
    default: return HB_ERR_INVALID;
  }
#undef HB_SURV
  count_launches(1);
  HB_LAUNCH_CHECK("nsga_survive");
  return HB_OK;
}

int launch_nsga_survive(const float *X, const float *F, const float *C, const float *FC, int64_t P, int64_t D, int64_t d,
                        float *Xn, float *Fn, float *Xcn, int32_t *Xen, cudaStream_t st) {
  return launch_nsga_survive_k(X, F, nullptr, C, FC, nullptr, P, D, d, 3, Xn, Fn, nullptr, Xcn, Xen, st);
}

}  // namespace hb
