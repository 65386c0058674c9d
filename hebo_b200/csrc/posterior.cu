// Posterior predict + MACE acquisition over candidate batches.
//   GP.predict   HEBO/hebo/models/gp/gp.py:137-164   mu = c + K* alpha ; var = s - ||Linv k*||^2 (floors, un-scaling)
//   MACE.eval    HEBO/hebo/acquisitions/acq.py:146-171  (LCB, -log EI, -log PI) with the log-approximation branch
//
// Three kernels per candidate chunk (chunked so the K* panel stays a bounded, L2-sized workspace):
//   kstar_kernel : raw candidates -> MinMax scale -> 1/lengthscale -> K* rows (and the K* alpha partial sums)
//   vnorm_kernel : V = K* Linv^T on the shared 128x128 SIMT GEMM core, triangular k-range, epilogue reduces
//                  ||v||^2 per row (V itself is never stored)
//   mace_kernel  : variance floors, un-scaling, MACE arithmetic (fp32, same operation order as the reference)
// All partial sums go to workspace slots and are combined in a fixed order: results are deterministic.
#include <stdlib.h>

#include "gemm_core.cuh"
#include "h16.cuh"
#include "kernels.h"

namespace hb {

constexpr int KS_ROWS = 32;     // candidates per CTA in kstar_kernel
constexpr int KS_COLS = 128;    // training points per sub-tile
constexpr int KS_GROUP = 512;   // training points per CTA (4 sub-tiles)
constexpr int KS_DC = 32;

// SPLIT: 0 = plain fp32 K* in KS (SIMT contraction / guard pass); 2 = the two-level fp16 split in the KS_lo buffer
// (h0 [mc_pad, np] halfs, then h1) and nothing else.
// fixlist != nullptr (SPLIT 0 only): the guard's second pass -- output row `slot` is the exact fp32 K* row of candidate
// fixlist[slot], for slot < *fixcount (blocks beyond the count exit at once); no mean partials.
// EMB: mixed model (gp_util.py:54-57): Zt holds d numeric rows followed by De embedding rows (both already divided by
// their lengthscales); the candidate's embedding features are gathered from tab_s (tables / le) by its categories
// Xe_s [m, e]; k* = s k_KERN(r over the numeric rows) Matern32(r over the embedding rows).
template <int KERN, int SPLIT, bool EMB>
__global__ void __launch_bounds__(256) kstar_kernel(const float *__restrict__ Xs, int64_t mc, int d,
                                                    const float *__restrict__ x_mul, const float *__restrict__ x_add,
                                                    const float *__restrict__ Zt, const float *__restrict__ alpha,
                                                    const float *__restrict__ hyp, int64_t n, int64_t np,
                                                    float *__restrict__ KS, float *__restrict__ KS_lo,
                                                    float *__restrict__ mupart, int64_t mc_pad,
                                                    const int32_t *__restrict__ fixlist, const int32_t *__restrict__ fixcount,
                                                    const int32_t *__restrict__ Xe_s, const float *__restrict__ tab_s,
                                                    ModelSpec sp) {
  extern __shared__ float zs[];                 // [d + De][KS_ROWS + 1] scaled candidates, transposed
  __shared__ __align__(16) float zt[KS_DC][KS_COLS];
  const int t = threadIdx.x;
  const int tx = t & 31, ty = t >> 5;           // warp ty owns rows ty*4..+3, lane tx owns cols tx*4..+3
  const int64_t r0 = (int64_t)blockIdx.x * KS_ROWS;
  const int64_t nrows = fixlist ? (int64_t)*fixcount : mc;
  if (r0 >= nrows) return;   // (block-uniform; only the guard pass launches more blocks than it needs)
  const float *ls = hyp + 3;
  for (int f = t; f < KS_ROWS * d; f += 256) {
    const int row = f / d, k = f - row * d;
    float z = 0.0f;
    if (r0 + row < nrows) {
      const int64_t src = fixlist ? (int64_t)fixlist[r0 + row] : r0 + row;
      const float x = Xs[src * d + k];
      float xt = __fadd_rn(__fmul_rn(x_mul[k], x), x_add[k]);   // TorchMinMaxScaler.transform, scalers.py:86-87
      if (sp.warp) xt = kumar_warp(xt, hyp[sp.h_wa() + k], hyp[sp.h_wb() + k]);   // input warp fused into the load stage
      z = xt * (1.0f / ls[k]);
    }
    zs[k * (KS_ROWS + 1) + row] = z;
  }
  const int De = EMB ? sp.De : 0;
  if (EMB) {
    for (int f = t; f < KS_ROWS * De; f += 256) {
      const int row = f / De, q = f - row * De;
      float z = 0.0f;
      if (r0 + row < nrows) {
        const int64_t src = fixlist ? (int64_t)fixlist[r0 + row] : r0 + row;
        const int c = sp.q_col[q];
        z = tab_s[sp.tab_off[c] + Xe_s[src * sp.e + c] * sp.emb_size[c] + sp.q_loc[q]];   // EmbTransform.forward, layers.py:33-34
      }
      zs[(d + q) * (KS_ROWS + 1) + row] = z;
    }
  }
  const float s = hyp[2];
  const float sa = pow2_scale(s, 1);   // fp16 operand scale: K* <= s lands in [0, 2)
  __half *KS_h0 = reinterpret_cast<__half *>(KS_lo), *KS_h1 = KS_h0 + mc_pad * np;
  float mu_acc[4] = {0.f, 0.f, 0.f, 0.f};
  const int64_t cg0 = (int64_t)blockIdx.y * KS_GROUP;
  for (int sub = 0; sub < KS_GROUP / KS_COLS; ++sub) {
    const int64_t c0 = cg0 + (int64_t)sub * KS_COLS;
    if (c0 >= np) break;
    float r2[4][4], r2e[4][4];   // (r2e dead unless EMB)
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) r2[i][j] = r2e[i][j] = 0.0f;
#pragma unroll
    for (int phase = 0; phase < (EMB ? 2 : 1); ++phase) {
      const int kbeg = phase ? d : 0, kend = phase ? d + De : d;
      float (&acc)[4][4] = phase ? r2e : r2;
      for (int k0 = kbeg; k0 < kend; k0 += KS_DC) {
        const int kc = min(KS_DC, kend - k0);
        __syncthreads();
        for (int f = t; f < kc * (KS_COLS / 4); f += 256) {
          const int kk = f >> 5, c4 = f & 31;
          *reinterpret_cast<float4 *>(&zt[kk][c4 * 4]) =
              __ldg(reinterpret_cast<const float4 *>(Zt + (int64_t)(k0 + kk) * np + c0 + c4 * 4));
        }
        __syncthreads();
#pragma unroll 4
        for (int kk = 0; kk < kc; ++kk) {
          const float4 b4 = *reinterpret_cast<const float4 *>(&zt[kk][tx * 4]);
          const float b[4] = {b4.x, b4.y, b4.z, b4.w};
          const float *zr = zs + (k0 + kk) * (KS_ROWS + 1) + ty * 4;
          const float a[4] = {zr[0], zr[1], zr[2], zr[3]};
#pragma unroll
          for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float df = a[i] - b[j];
              acc[i][j] = fmaf(df, df, acc[i][j]);
            }
        }
      }
    }
    const float4 al4 = __ldg(reinterpret_cast<const float4 *>(alpha + c0 + tx * 4));
    const float al[4] = {al4.x, al4.y, al4.z, al4.w};
    // pad columns (training index >= n) must come out as exact zeros: the pad block of Linv is the identity.  Only the
    // last 128-column sub-tile can contain them, so the test is hoisted out of the per-pair code.
    const int ncol = (int)min((int64_t)4, max((int64_t)0, n - (c0 + tx * 4)));   // valid columns among this thread's 4
    const int64_t rowoff = (r0 + ty * 4) * np + c0 + tx * 4;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float o[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float kv = s * kern_eval<KERN>(r2[i][j]);
        if (EMB) kv *= kern_eval<HB_KERN_MATERN32>(r2e[i][j]);
        if (j >= ncol) kv = 0.0f;
        o[j] = kv;
        mu_acc[i] = fmaf(kv, al[j], mu_acc[i]);
      }
      const int64_t off = rowoff + (int64_t)i * np;
      if (SPLIT == 2) {
        unsigned int a01, a23, b01, b23;
        split_h16x2(o[0] * sa, o[1] * sa, a01, b01);
        split_h16x2(o[2] * sa, o[3] * sa, a23, b23);
        *reinterpret_cast<uint2 *>(KS_h0 + off) = make_uint2(a01, a23);
        *reinterpret_cast<uint2 *>(KS_h1 + off) = make_uint2(b01, b23);
      } else {
        *reinterpret_cast<float4 *>(KS + off) = make_float4(o[0], o[1], o[2], o[3]);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float v = warp_sum(mu_acc[i]);
    if (tx == 0 && mupart) mupart[(int64_t)blockIdx.y * mc_pad + r0 + ty * 4 + i] = v;
  }
}

// ||Linv k*||^2 per candidate and column tile J:  vpart[J][row] = sum_{c in tile J} (sum_{k <= c} KS[row][k] Linv[c][k])^2
__global__ void __launch_bounds__(GTHREADS, 2) vnorm_kernel(const float *__restrict__ KS, const float *__restrict__ Linv,
                                                            int64_t np, int64_t mc_pad, float *__restrict__ vpart) {
  __shared__ GemmSmem sm;
  const int nt = (int)(np / GT);
  const int J = nt - 1 - (int)blockIdx.x;   // heaviest (longest k range) tiles first
  const int64_t rt = blockIdx.y;
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.0f;
  gemm_mainloop<true, true>(KS + rt * GT * np, np, Linv + (int64_t)J * GT * np, np, 0, (J + 1) * GT, acc, sm);
  const int tx = threadIdx.x & 15;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    float s = 0.0f;
#pragma unroll
    for (int j = 0; j < 8; ++j) s = fmaf(acc[i][j], acc[i][j], s);
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (tx == 0) vpart[(int64_t)J * mc_pad + rt * GT + gemm_row(i)] = s;
  }
}

// ---- precision guard of the tensor path ------------------------------------------------------------------
// sigma^2 = s - ||v||^2 cancels when a candidate sits on the data; the tensor cores' fp32 accumulation in TMEM is
// not round-to-nearest (measured ~5e-6 relative on ||v||^2), which would exceed the 1e-4 sigma criterion once
// sigma^2 < ~s/40.  Rows whose variance falls below theta * s (default 0.12) are therefore flagged and their ||v||^2 is
// recomputed on the FP32 SIMT pipe from the same operands (K* = hi + lo); typical BO batches flag few rows, a
// batch that sits entirely on the data degrades gracefully to the SIMT contraction.
static float guard_theta() {   // HEBO_B200_GUARD_THETA overrides (0 disables the guard: measurement only)
  static float v = -1.0f;
  if (v < 0.0f) {
    const char *e = getenv("HEBO_B200_GUARD_THETA");
    v = e ? (float)atof(e) : 0.12f;
  }
  return v;
}

// measurement hook (bench.py "guard_flagged_frac"): rows seen / rows flagged by the guard since the last reset
__device__ unsigned long long g_guard_stats[2];

__global__ void __launch_bounds__(256) guard_kernel(const float *__restrict__ vpart, int nslots, int64_t mc,
                                                    int64_t mc_pad, const float *__restrict__ hyp,
                                                    float theta, int32_t *__restrict__ fixmap,
                                                    int32_t *__restrict__ fixlist, int32_t *__restrict__ count) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= mc) return;
  const float s = hyp[2];
  float vsq = 0.0f;
  for (int j = 0; j < nslots; ++j) vsq += vpart[(int64_t)j * mc_pad + r];
  int32_t slot = -1;
  if ((s - vsq) < theta * s) {
    slot = atomicAdd(count, 1);
    fixlist[slot] = (int32_t)r;
    atomicAdd(&g_guard_stats[1], 1ull);
  }
  fixmap[r] = slot;
  if (threadIdx.x == 0) atomicAdd(&g_guard_stats[0], (unsigned long long)min((int64_t)blockDim.x, mc - (int64_t)blockIdx.x * blockDim.x));
}

int guard_stats(unsigned long long *out, int reset) {
  HB_CUDA(cudaMemcpyFromSymbol(out, g_guard_stats, 2 * sizeof(unsigned long long)));
  if (reset) {
    const unsigned long long z[2] = {0ull, 0ull};
    HB_CUDA(cudaMemcpyToSymbol(g_guard_stats, z, sizeof(z)));
  }
  return HB_OK;
}

__global__ void __launch_bounds__(GTHREADS, 1) vnorm_fix_kernel(const float *__restrict__ KS_hi,
                                                                const float *__restrict__ KS_lo,
                                                                const float *__restrict__ Linv, int64_t np,
                                                                int64_t mc_pad, const int32_t *__restrict__ fixlist,
                                                                const int32_t *__restrict__ count,
                                                                float *__restrict__ vfix, int compact) {
  __shared__ GemmSmem sm;
  const int cnt = *count;
  const int64_t g = blockIdx.y;
  if (g * GT >= cnt) return;
  const int nt = (int)(np / GT);
  const int J = nt - 1 - (int)blockIdx.x;
  int64_t rows[2];
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const int64_t slot = g * GT + ((threadIdx.x + q * GTHREADS) >> 2);
    rows[q] = compact ? (slot < cnt ? slot : 0) : fixlist[slot < cnt ? slot : 0];   // compact: KS_hi row = slot
  }
  double acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.0;
  gemm_mainloop_gatherA(KS_hi, KS_lo, np, rows, Linv + (int64_t)J * GT * np, np, 0, (J + 1) * GT, acc, sm);
  const int tx = threadIdx.x & 15;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    double s = 0.0;
#pragma unroll
    for (int j = 0; j < 8; ++j) s = fma(acc[i][j], acc[i][j], s);
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (tx == 0) vfix[(int64_t)J * mc_pad + g * GT + gemm_row(i)] = (float)s;
  }
}

// ---- Philox4x32-10 + Box-Muller for the production (non-parity) noise path
__device__ __forceinline__ void philox_round(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
  const uint32_t hi0 = __umulhi(M0, c[0]), lo0 = M0 * c[0];
  const uint32_t hi1 = __umulhi(M1, c[2]), lo1 = M1 * c[2];
  const uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
  c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
}
__device__ __forceinline__ void philox_normal2(uint64_t seed, uint64_t row, float &z0, float &z1) {
  uint32_t c[4] = {(uint32_t)row, (uint32_t)(row >> 32), 0u, 0u};
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    philox_round(c, k0, k1);
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  const float u0 = ((float)c[0] + 0.5f) * 2.3283064365386963e-10f;   // (0,1)
  const float u1 = ((float)c[1] + 0.5f) * 2.3283064365386963e-10f;
  const float rad = sqrtf(-2.0f * logf(u0));
  float sn, cs;
  sincospif(2.0f * u1, &sn, &cs);
  z0 = rad * cs;
  z1 = rad * sn;
}

// MACE.eval arithmetic for one row (acq.py:151-171), fp32, same operation order as the reference
__device__ __forceinline__ void mace_row(float py, float ps2, float noise_var, float tau, float kappa, float eps,
                                         float z1, float z2, float &lcb, float &o1, float &o2) {
  const float noise = __fmul_rn(1.4142135623730951f, sqrtf(noise_var));      // acq.py:152
  const float ps = fmaxf(sqrtf(ps2), 1.1920929e-07f);                        // acq.py:153
  lcb = __fsub_rn(__fadd_rn(py, __fmul_rn(noise, z1)), __fmul_rn(kappa, ps));   // acq.py:154
  const float num = __fsub_rn(__fsub_rn(__fsub_rn(tau, eps), py), __fmul_rn(noise, z2));
  const float zz = __fdiv_rn(num, ps);                                       // acq.py:155
  const float zsq = __fmul_rn(zz, zz);
  const float log_phi = __fsub_rn(__fdiv_rn(-zsq, 2.0f), 0.9189385332046727f);   // Normal.log_prob
  const float Phi = __fmul_rn(0.5f, __fadd_rn(1.0f, erff(__fdiv_rn(zz, 1.4142135623730951f))));   // Normal.cdf
  const float EI = __fmul_rn(ps, __fadd_rn(__fmul_rn(Phi, zz), expf(log_phi)));   // acq.py:160
  const float logEI = logf(EI), logPI = logf(Phi);
  const bool ok = (zz > -6.0f) && isfinite(logEI) && isfinite(logPI);        // acq.py:164
  if (ok) {
    o1 = -logEI;
    o2 = -logPI;
  } else {
    const float half_z2 = __fmul_rn(0.5f, zsq);
    const float logEIapp = __fsub_rn(__fsub_rn(logf(ps), half_z2), logf(__fsub_rn(zsq, 1.0f)));     // acq.py:161
    const float logPIapp = __fsub_rn(__fsub_rn(-half_z2, logf(-zz)), 0.9189385332046727f);          // acq.py:162
    o1 = -logEIapp;
    o2 = -logPIapp;
  }
}

// standalone epilogue: MACE over any model's (mu, var) already on the device
__global__ void __launch_bounds__(256) mace_only_kernel(const float *__restrict__ mu, const float *__restrict__ var,
                                                        int64_t m, float noise_var, float tau, float kappa, float eps,
                                                        const float *__restrict__ xi1, const float *__restrict__ xi2,
                                                        uint64_t seed, float *__restrict__ F) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= m) return;
  float z1, z2;
  if (xi1 && xi2) {
    z1 = xi1[r];
    z2 = xi2[r];
  } else {
    philox_normal2(seed, (uint64_t)r, z1, z2);
  }
  float lcb, o1, o2;
  mace_row(mu[r], var[r], noise_var, tau, kappa, eps, z1, z2, lcb, o1, o2);
  F[r * 3 + 0] = lcb;
  F[r * 3 + 1] = o1;
  F[r * 3 + 2] = o2;
}

int launch_mace_only(const float *mu, const float *var, int64_t m, float noise_var, float tau, float kappa, float eps,
                     const float *xi1, const float *xi2, uint64_t seed, float *F, cudaStream_t st) {
  if (m <= 0) return HB_ERR_INVALID;
  mace_only_kernel<<<(int)ceil_div(m, 256), 256, 0, st>>>(mu, var, m, noise_var, tau, kappa, eps, xi1, xi2, seed, F);
  count_launches(1);
  HB_LAUNCH_CHECK("mace_only");
  return HB_OK;
}


__global__ void __launch_bounds__(256) mace_kernel(const float *__restrict__ mupart, int ncg,
                                                   const float *__restrict__ vpart, int nt,
                                                   const int32_t *__restrict__ fixmap,
                                                   const float *__restrict__ vfix, int nt_fix, int64_t mc,
                                                   int64_t mc_pad, int64_t row_offset, int64_t rng_offset,
                                                   const float *__restrict__ hyp, float y_mean, float y_std,
                                                   int pred_likeli, float tau, float kappa, float eps,
                                                   const float *__restrict__ xi1, const float *__restrict__ xi2,
                                                   uint64_t seed, float *__restrict__ F, float *__restrict__ mu_out,
                                                   float *__restrict__ var_out) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= mc) return;
  const float sn2 = hyp[0], c = hyp[1], s = hyp[2];
  float mu_t = 0.0f;
  for (int g = 0; g < ncg; ++g) mu_t += mupart[(int64_t)g * mc_pad + r];
  mu_t += c;
  float vsq = 0.0f;
  const int fm = fixmap ? fixmap[r] : -1;
  if (fm >= 0) {
    for (int j = 0; j < nt_fix; ++j) vsq += vfix[(int64_t)j * mc_pad + fm];     // guarded row: FP32 SIMT recomputation
  } else {
    for (int j = 0; j < nt; ++j) vsq += vpart[(int64_t)j * mc_pad + r];
  }
  float var_t = s - vsq;
  if (pred_likeli) var_t += sn2;                            // gp.py:158-159: pred = lik(pred) adds the noise FIRST,
  var_t = fmaxf(var_t, 1e-6f);                              // then .variance applies gpytorch's min_variance floor (fp32)
  const float py = __fadd_rn(__fmul_rn(mu_t, y_std), y_mean);                 // gp.py:162
  const float ps2 = fmaxf(__fmul_rn(var_t, __fmul_rn(y_std, y_std)), 1.1920929e-07f);   // gp.py:163-164
  const int64_t gr = row_offset + r;
  if (mu_out) mu_out[gr] = py;
  if (var_out) var_out[gr] = ps2;
  if (!F) return;
  // ---- MACE, acq.py:151-171
  float z1, z2;
  if (xi1 && xi2) {
    z1 = xi1[gr];
    z2 = xi2[gr];
  } else {
    philox_normal2(seed, (uint64_t)(rng_offset + gr), z1, z2);
  }
  const float noise_var = __fmul_rn(sn2, __fmul_rn(y_std, y_std));           // gp.py:184
  float lcb, o1, o2;
  mace_row(py, ps2, noise_var, tau, kappa, eps, z1, z2, lcb, o1, o2);
  F[gr * 3 + 0] = lcb;
  F[gr * 3 + 1] = o1;
  F[gr * 3 + 2] = o2;
}

// ---- GeneralAcq.eval (acq.py:233-242) over O = num_obj + num_constr outputs, fp32, the reference's operation order:
//   ps = sqrt(ps2).clamp(min = eps) ; py += sqrt(noise) * xi (use_noise) ; out = py - kappa ps (objectives) | - c_kappa ps
// mu / var [O, m] output-major (O calls of the posterior, one output row each); out [m, O] row-major like the reference's
// `out`; cv [m] (optional) = sum_j max(0, out[:, num_obj + j]) in ascending j, pymoo 0.6 calc_cv as recalled (NaN
// propagates).  xi [m, O] = the reference's single torch.randn(py.shape) draw, or NULL: Philox normals keyed by
// (seed, rng_offset + row, output), the pair (2 j, 2 j + 1) from counter word j -- with O <= 2 the draws of mace_kernel.
__device__ __forceinline__ void philox_normal2_word(uint64_t seed, uint64_t row, uint32_t word, float &z0, float &z1) {
  uint32_t c[4] = {(uint32_t)row, (uint32_t)(row >> 32), word, 0u};
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    philox_round(c, k0, k1);
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  const float u0 = ((float)c[0] + 0.5f) * 2.3283064365386963e-10f;   // (0,1)
  const float u1 = ((float)c[1] + 0.5f) * 2.3283064365386963e-10f;
  const float rad = sqrtf(-2.0f * logf(u0));
  float sn, cs;
  sincospif(2.0f * u1, &sn, &cs);
  z0 = rad * cs;
  z1 = rad * sn;
}

__global__ void __launch_bounds__(256) general_acq_kernel(const float *__restrict__ mu, const float *__restrict__ var, int64_t m,
                                                          int num_obj, int O, const float *__restrict__ noise_var, float kappa,
                                                          float c_kappa, int use_noise, const float *__restrict__ xi,
                                                          uint64_t seed, int64_t rng_offset, float *__restrict__ out,
                                                          float *__restrict__ cv) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= m) return;
  float cvs = 0.0f, z1 = 0.0f;
  for (int o = 0; o < O; ++o) {
    float py = mu[(int64_t)o * m + r];
    const float s = sqrtf(var[(int64_t)o * m + r]);
    const float ps = isnan(s) ? s : fmaxf(s, 1.1920929e-07f);                // clamp(min = finfo.eps) keeps a NaN
    if (use_noise) {
      float z;
      if (xi) {
        z = xi[r * O + o];
      } else if ((o & 1) == 0) {
        philox_normal2_word(seed, (uint64_t)(rng_offset + r), (uint32_t)(o >> 1), z, z1);
      } else {
        z = z1;
      }
      py = __fadd_rn(py, __fmul_rn(sqrtf(noise_var[o]), z));                  // acq.py:236-238
    }
    const float v = __fsub_rn(py, __fmul_rn(o < num_obj ? kappa : c_kappa, ps));   // acq.py:240-241
    out[r * O + o] = v;
    if (o >= num_obj) cvs = __fadd_rn(cvs, v > 0.0f ? v : (isnan(v) ? v : 0.0f));
  }
  if (cv) cv[r] = cvs;
}

int launch_general_acq(const float *mu, const float *var, int64_t m, int num_obj, int num_constr, const float *noise_var,
                       float kappa, float c_kappa, int use_noise, const float *xi, uint64_t seed, int64_t rng_offset, float *out,
                       float *cv, cudaStream_t st) {
  if (m <= 0 || num_obj < 1 || num_obj > 8 || num_constr < 0 || num_obj + num_constr > 64) return HB_ERR_INVALID;
  general_acq_kernel<<<(int)ceil_div(m, 256), 256, 0, st>>>(mu, var, m, num_obj, num_obj + num_constr, noise_var, kappa, c_kappa,
                                                            use_noise, xi, seed, rng_offset, out, cv);
  count_launches(1);
  HB_LAUNCH_CHECK("general_acq");
  return HB_OK;
}

int kstar_groups(int64_t np) { return (int)ceil_div(np, KS_GROUP); }

// plain fp32 K* rows + mean partials (posterior_grad.cu)
int launch_kstar_plain(const float *xs, const int32_t *xe, int64_t mc, const ModelSpec &sp, const float *tab_s,
                       const float *x_mul, const float *x_add, const float *Zt,
                       const float *alpha, const float *hyp, int64_t n, int64_t np, int kern, float *KS, float *mupart,
                       int64_t mc_pad, cudaStream_t st) {
  const int d = sp.d;
  const size_t dyn = (size_t)sp.dtot() * (KS_ROWS + 1) * sizeof(float);
  if (dyn > 30 * 1024) return HB_ERR_INVALID;
  const dim3 g1((unsigned)ceil_div(mc, KS_ROWS), (unsigned)kstar_groups(np));
#define HB_KP(K)                                                                                                              \
  do {                                                                                                                        \
    if (sp.e > 0)                                                                                                             \
      kstar_kernel<K, 0, true><<<g1, 256, dyn, st>>>(xs, mc, d, x_mul, x_add, Zt, alpha, hyp, n, np, KS, nullptr, mupart,     \
                                                     mc_pad, nullptr, nullptr, xe, tab_s, sp);                               \
    else                                                                                                                      \
      kstar_kernel<K, 0, false><<<g1, 256, dyn, st>>>(xs, mc, d, x_mul, x_add, Zt, alpha, hyp, n, np, KS, nullptr, mupart,    \
                                                      mc_pad, nullptr, nullptr, nullptr, nullptr, sp);                       \
  } while (0)
  if (kern == HB_KERN_MATERN32) HB_KP(0); else if (kern == HB_KERN_MATERN52) HB_KP(1); else HB_KP(2);
#undef HB_KP
  count_launches(1);
  return HB_OK;
}

size_t posterior_ws_bytes(int64_t np, int64_t d, int64_t m_chunk) {
  const int64_t mc_pad = round_up(m_chunk, 2 * GT);
  const int64_t ncg = ceil_div(np, KS_GROUP);
  const int64_t nt = np / GT;
  return (size_t)(2 * mc_pad * np + ncg * mc_pad + 2 * nt * mc_pad + 2 * mc_pad) * sizeof(float) + 512;
}

int launch_posterior_mace(const float *Xs, const int32_t *Xe_s, int64_t m, int64_t rng_offset, int64_t n, int64_t np, const ModelSpec &sp,
                          const float *tab_s, const float *x_mul,
                          const float *x_add, const float *Zt, const float *alpha, const float *Linv,
                          const float *Linv_hi, const float *Linv_lo, const float *hyp, int kern, float y_mean, float y_std, int pred_likeli, float tau,
                          float kappa, float eps, const float *xi1, const float *xi2, uint64_t seed, float *F,
                          float *mu, float *var, void *ws, int64_t ws_bytes, int64_t m_chunk, cudaStream_t st) {
  const int64_t d = sp.d;
  if (m <= 0 || n <= 0 || sp.dtot() <= 0 || np % GT != 0 || n > np || m_chunk <= 0) return HB_ERR_INVALID;
  if (kern < 0 || kern > 2 || (sp.e > 0 && (!Xe_s || !tab_s))) return HB_ERR_INVALID;
  if ((size_t)ws_bytes < posterior_ws_bytes(np, d, m_chunk)) return HB_ERR_INVALID;
  const size_t dyn = (size_t)sp.dtot() * (KS_ROWS + 1) * sizeof(float);
  if (dyn > 30 * 1024) return HB_ERR_INVALID;   // d + De <= 232 with the static 16 KB tile
  const int64_t mc_pad_max = round_up(m_chunk, 2 * GT);   // 256: one CTA pair of the 2-SM tensor path
  const int ncg = (int)ceil_div(np, KS_GROUP);
  const int nt = (int)(np / GT);
  const bool tensor = Linv_hi != nullptr && Linv_lo != nullptr;   // tcgen05 path (two-level fp16 split), else FP32 SIMT
  const bool h16 = tensor;
  // workspace: the K* chunk (KS: fp32 rows of the SIMT / guard passes; KS2: the fp16 two-level split h0 | h1 of the
  // tensor path), the mean partials and the per-chunk partial-sum buffers.  (Building chunk i+1 on a side stream under
  // the tensor-core contraction of chunk i was measured and dropped: the contraction draws ~all of the L2 -> SM
  // bandwidth, the co-running CUDA-core kernel slowed it by 30 %.)
  float *KS = reinterpret_cast<float *>(ws);
  float *KS2 = KS + mc_pad_max * np;
  float *mupart = KS2 + mc_pad_max * np;
  float *vpart = mupart + (int64_t)ncg * mc_pad_max;
  float *vfix = vpart + (int64_t)nt * mc_pad_max;
  int32_t *fixmap = reinterpret_cast<int32_t *>(vfix + (int64_t)nt * mc_pad_max);
  int32_t *fixlist = fixmap + mc_pad_max;
  int32_t *fixcount = fixlist + mc_pad_max;
  for (int64_t c0 = 0; c0 < m; c0 += m_chunk) {
    const int64_t mc = min(m_chunk, m - c0);
    const int64_t mc_pad = round_up(mc, GT);
    const cudaStream_t ks_st = st;
    const dim3 g1((unsigned)ceil_div(mc, KS_ROWS), (unsigned)ncg);
    const float *xs = Xs + c0 * d;
    const int32_t *xe = sp.e > 0 ? Xe_s + c0 * sp.e : nullptr;
#define HB_KSTAR(K, S)                                                                                                          \
  do {                                                                                                                          \
    if (sp.e > 0)                                                                                                               \
      kstar_kernel<K, S, true><<<g1, 256, dyn, ks_st>>>(xs, mc, (int)d, x_mul, x_add, Zt, alpha, hyp, n, np, KS, KS2, mupart,   \
                                                        mc_pad_max, nullptr, nullptr, xe, tab_s, sp);                          \
    else                                                                                                                        \
      kstar_kernel<K, S, false><<<g1, 256, dyn, ks_st>>>(xs, mc, (int)d, x_mul, x_add, Zt, alpha, hyp, n, np, KS, KS2, mupart,  \
                                                         mc_pad_max, nullptr, nullptr, nullptr, nullptr, sp);                  \
  } while (0)
    if (h16) {
      if (kern == HB_KERN_MATERN32) HB_KSTAR(0, 2); else if (kern == HB_KERN_MATERN52) HB_KSTAR(1, 2); else HB_KSTAR(2, 2);
    } else {
      if (kern == HB_KERN_MATERN32) HB_KSTAR(0, 0); else if (kern == HB_KERN_MATERN52) HB_KSTAR(1, 0); else HB_KSTAR(2, 0);
    }
#undef HB_KSTAR
    int nslots = nt;
    if (tensor) {
      const __half *kh0 = reinterpret_cast<const __half *>(KS2), *kh1 = kh0 + mc_pad_max * np;
      const int s = launch_vnorm_h16(kh0, kh1, mc_pad_max, reinterpret_cast<const __half *>(Linv_hi),
                                     reinterpret_cast<const __half *>(Linv_lo), Linv_lo + np * np / 2, hyp, np, round_up(mc, 2 * GT),
                                     mc_pad_max, vpart, st);
      if (s != HB_OK) return s;
      nslots = (int)ceil_div(np, 256);
      HB_CUDA(cudaMemsetAsync(fixcount, 0, sizeof(int32_t), st));
      guard_kernel<<<(int)ceil_div(mc, 256), 256, 0, st>>>(vpart, nslots, mc, mc_pad_max, hyp, guard_theta(), fixmap, fixlist, fixcount);
      const dim3 gf((unsigned)nt, (unsigned)(mc_pad / GT));
      {   // exact fp32 K* rows of the flagged candidates only (compact, row = slot), then their FP32 contraction
#define HB_KFIX(K)                                                                                                              \
  do {                                                                                                                          \
    if (sp.e > 0)                                                                                                               \
      kstar_kernel<K, 0, true><<<g1, 256, dyn, st>>>(xs, mc, (int)d, x_mul, x_add, Zt, alpha, hyp, n, np, KS, nullptr, nullptr, \
                                                     mc_pad_max, fixlist, fixcount, xe, tab_s, sp);                            \
    else                                                                                                                        \
      kstar_kernel<K, 0, false><<<g1, 256, dyn, st>>>(xs, mc, (int)d, x_mul, x_add, Zt, alpha, hyp, n, np, KS, nullptr, nullptr,\
                                                      mc_pad_max, fixlist, fixcount, nullptr, nullptr, sp);                    \
  } while (0)
        if (kern == HB_KERN_MATERN32) HB_KFIX(0); else if (kern == HB_KERN_MATERN52) HB_KFIX(1); else HB_KFIX(2);
#undef HB_KFIX
        count_launches(1);
      }
      vnorm_fix_kernel<<<gf, GTHREADS, 0, st>>>(KS, nullptr, Linv, np, mc_pad_max, fixlist, fixcount, vfix, 1);
      count_launches(4);
    } else {
      const dim3 g2((unsigned)nt, (unsigned)(mc_pad / GT));
      prof_begin(st);
      vnorm_kernel<<<g2, GTHREADS, 0, st>>>(KS, Linv, np, mc_pad_max, vpart);
      prof_end(st);
      count_launches(3);
    }
    mace_kernel<<<(int)ceil_div(mc, 256), 256, 0, st>>>(mupart, ncg, vpart, nslots, tensor ? fixmap : nullptr, vfix, nt, mc,
                                                        mc_pad_max, c0, rng_offset, hyp, y_mean, y_std,
                                                        pred_likeli, tau, kappa, eps, xi1, xi2, seed, F, mu, var);
  }
  HB_LAUNCH_CHECK("posterior_mace");
  return HB_OK;
}

}  // namespace hb
