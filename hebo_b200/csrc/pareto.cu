// K-objective constrained non-dominated filter (all objectives minimised, 1 <= K <= 8): the rank-0 set that pymoo's NSGA-II
// hands back as res.X in HEBO/hebo/acq_optimizers/evolution_optimizer.py:141-149, computed exactly on the device for
// candidate batches of any size.  F is read with a row stride ldf >= K, so the objective columns of a wider [m, O]
// acquisition output (GeneralAcq: objectives first, then constraints) are filtered in place.
//
//   a dominates b  <=>  all(a <= b) and any(a < b)
// A row with a NaN objective never dominates (every comparison is false) and is EXCLUDED from the front: it cannot be
// dominated either, and the selection step (hebo.py:182-193) must never be handed a candidate whose acquisition is NaN.
// With a constraint violation cv [m] (cv = sum_j max(0, g_j), pymoo 0.6 calc_cv as recalled -- pymoo is not installed)
// only FEASIBLE rows (cv <= 0; a NaN cv is never feasible) take part: an infeasible row is loaded as NaN, so it neither
// dominates nor survives.  If no row is feasible, the result is the single row of least cv (lowest index on ties, rows
// with a NaN objective or cv never chosen) -- the least_infeasible rule of pymoo's filter_optimum behind res.X -- found
// with one 64-bit atomicMin on the device, without a host read.
//
// m <= 4096: one tiled all-pairs pass.  Larger m: (1) exact front FS of a stratified sample (strided_row), (2) every point is
// tested against FS only (anything FS dominates is dominated in the full set), (3) exact all-pairs among the
// survivors.  By transitivity of dominance (restricted to the feasible rows, for any K) step 3 sees every true dominator,
// so the result is exact.  Compaction is order preserving (count / scan / scatter), so idx_out is ascending and
// deterministic.  hb_pareto_front3 is the K = 3, ldf = 3, cv = NULL instantiation of this one code path.
#include "kernels.h"

namespace hb {

constexpr int PB = 256;
constexpr int PARETO_DIRECT_MAX = 4096;    // above: sample front -> filter all -> exact among survivors (93 us vs 784 us at m = 16k)
constexpr int PARETO_SAMPLE = 4096;

// Row of the a-th element of a strided (sample) list: one row out of every aligned block of `stride` consecutive rows, at a
// hashed offset inside the block.  A plain a * stride sample of a Sobol candidate batch (HEBO's quasi_sample, hebo.py:99-113)
// is confined to a thin slab of the box (indices = 0 mod 2^k fix the leading k digits of the first coordinates), its front
// dominated almost nothing outside the slab and stage 3 saw 12-23 k survivors (1.3 ms instead of 0.1 ms, seed dependent:
// the rank skew of the 8-GPU run); the hashed offset leaves 4-21.  Any sample keeps the result exact.
__device__ __forceinline__ int64_t strided_row(int a, int stride) {
  if (stride <= 1) return a;
  const uint32_t h = ((uint32_t)a * 2654435761u) >> 11;
  return (int64_t)a * stride + (int64_t)(h % (uint32_t)stride);
}

// flags[a] := 0 if list-A element a is dominated by an element of list B (or carries a NaN, or is infeasible); flags must be
// preset to 1.  idxA / idxB == nullptr -> identity lists of length *nA / *nB (or the host bounds when the count pointers are
// null).  gridDim.y splits list B into segments (each block tests its 256 A rows against one segment and only ever CLEARS
// flags: idempotent, no ordering needed), so a short list A against a long list B -- the 4096 x 4096 sample-front pass, 16
// blocks and 205 us when B was walked by one block per A tile -- still fills the machine.
template <int K>
__global__ void __launch_bounds__(PB) nondominated_kernel(const float *__restrict__ F, int64_t ldf, const float *__restrict__ cv,
                                                          const int32_t *__restrict__ idxA,
                                                          const int32_t *__restrict__ nA_ptr, int nA_host, int strideA,
                                                          const int32_t *__restrict__ idxB,
                                                          const int32_t *__restrict__ nB_ptr, int nB_host, int strideB,
                                                          uint8_t *__restrict__ flags) {
  __shared__ float bs[K][PB];
  const int nA = nA_ptr ? *nA_ptr : nA_host;
  const int nB = nB_ptr ? *nB_ptr : nB_host;
  if ((int)(blockIdx.x * PB) >= nA) return;
  const int seg = (int)ceil_div(ceil_div(nB, (int64_t)gridDim.y), PB) * PB;      // segment length, multiple of the tile
  const int jbeg = blockIdx.y * seg, jend = min(nB, jbeg + seg);
  const int a = blockIdx.x * PB + threadIdx.x;
  const bool active = a < nA;
  float av[K];
  bool dominated = !active;
#pragma unroll
  for (int k = 0; k < K; ++k) av[k] = 0.f;
  if (active) {
    const int64_t ia = idxA ? idxA[a] : strided_row(a, strideA);
#pragma unroll
    for (int k = 0; k < K; ++k) {
      av[k] = F[ia * ldf + k];
      dominated |= isnan(av[k]);
    }
    if (cv) dominated |= !(cv[ia] <= 0.f);
  }
  for (int j0 = jbeg; j0 < jend; j0 += PB) {
    const int j = j0 + threadIdx.x;
    if (j < jend) {
      const int64_t ib = idxB ? idxB[j] : strided_row(j, strideB);
      const bool feasible = !cv || cv[ib] <= 0.f;
#pragma unroll
      for (int k = 0; k < K; ++k) bs[k][threadIdx.x] = feasible ? F[ib * ldf + k] : NAN;
    }
    __syncthreads();
    const int lim = min(PB, jend - j0);
    if (!dominated) {
      for (int u = 0; u < lim; ++u) {
        bool le = true, lt = false;
#pragma unroll
        for (int k = 0; k < K; ++k) {
          const float x = bs[k][u];
          le &= x <= av[k];
          lt |= x < av[k];
        }
        if (le & lt) {
          dominated = true;
          break;
        }
      }
    }
    if (__syncthreads_and(dominated)) break;
  }
  if (active && dominated) flags[a] = 0;
}

// least-infeasible candidate: key = (float bits of cv) << 32 | row, over the rows without a NaN objective or cv (cv >= 0 as
// a sum of max(0, g), so the float bits order like the values)
template <int K>
__global__ void __launch_bounds__(PB) least_cv_kernel(const float *__restrict__ F, int64_t ldf, const float *__restrict__ cv,
                                                      int m, unsigned long long *__restrict__ key) {
  const int r = blockIdx.x * PB + threadIdx.x;
  unsigned long long mine = ~0ull;
  if (r < m) {
    const float c = cv[r];
    bool ok = !isnan(c);
#pragma unroll
    for (int k = 0; k < K; ++k) ok &= !isnan(F[(int64_t)r * ldf + k]);
    if (ok) mine = ((unsigned long long)__float_as_uint(fmaxf(c, 0.0f)) << 32) | (unsigned)r;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mine = min(mine, __shfl_xor_sync(0xffffffffu, mine, o));
  if ((threadIdx.x & 31) == 0 && mine != ~0ull) atomicMin(key, mine);
}

// no feasible row -> the front is the least-infeasible row
__global__ void least_cv_apply_kernel(const unsigned long long *__restrict__ key, int32_t *__restrict__ idx_out,
                                      int32_t *__restrict__ count) {
  if (*count == 0 && *key != ~0ull) {
    idx_out[0] = (int32_t)(*key & 0xffffffffull);
    *count = 1;
  }
}

// order-preserving compaction of list A by flags: count -> scan -> scatter
__global__ void __launch_bounds__(PB) compact_count_kernel(const uint8_t *__restrict__ flags,
                                                           const int32_t *__restrict__ nA_ptr, int nA_host,
                                                           int32_t *__restrict__ block_counts) {
  const int nA = nA_ptr ? *nA_ptr : nA_host;
  const int a = blockIdx.x * PB + threadIdx.x;
  const int keep = (a < nA) ? flags[a] : 0;
  const int c = __syncthreads_count(keep);
  if (threadIdx.x == 0) block_counts[blockIdx.x] = c;
}

__global__ void __launch_bounds__(1024) compact_scan_kernel(int32_t *__restrict__ block_counts, int nblocks,
                                                            int32_t *__restrict__ total) {
  // exclusive scan in place (single block, sequential over 1024-wide strips)
  __shared__ int32_t sh[1024];
  __shared__ int32_t carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int base = 0; base < nblocks; base += 1024) {
    const int i = base + threadIdx.x;
    const int v = (i < nblocks) ? block_counts[i] : 0;
    sh[threadIdx.x] = v;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
      const int add = (threadIdx.x >= (unsigned)o) ? sh[threadIdx.x - o] : 0;
      __syncthreads();
      sh[threadIdx.x] += add;
      __syncthreads();
    }
    const int incl = sh[threadIdx.x];
    if (i < nblocks) block_counts[i] = carry + incl - v;
    __syncthreads();
    if (threadIdx.x == 1023) carry += incl;
    __syncthreads();
  }
  if (threadIdx.x == 0) *total = carry;
}

__global__ void __launch_bounds__(PB) compact_scatter_kernel(const uint8_t *__restrict__ flags,
                                                             const int32_t *__restrict__ idxA,
                                                             const int32_t *__restrict__ nA_ptr, int nA_host,
                                                             int strideA, const int32_t *__restrict__ block_offsets,
                                                             int32_t *__restrict__ out_idx) {
  __shared__ int32_t warp_tot[PB / 32];
  const int nA = nA_ptr ? *nA_ptr : nA_host;
  const int a = blockIdx.x * PB + threadIdx.x;
  const int keep = (a < nA) ? flags[a] : 0;
  const unsigned bal = __ballot_sync(0xffffffffu, keep);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int pre = __popc(bal & ((1u << lane) - 1u));
  if (lane == 0) warp_tot[warp] = __popc(bal);
  __syncthreads();
  int woff = 0;
  for (int w = 0; w < warp; ++w) woff += warp_tot[w];
  if (keep) {
    const int32_t src = idxA ? idxA[a] : (int32_t)strided_row(a, strideA);
    out_idx[block_offsets[blockIdx.x] + woff + pre] = src;
  }
}

struct ParetoWs {
  uint8_t *flags;
  int32_t *counts;   // block counts / offsets
  int32_t *listA;    // survivors after stage 2
  int32_t *listS;    // sample front
  int32_t *nS;
  int32_t *nA;
  unsigned long long *key;   // least-infeasible row (inside the nS slot's padding)
};

static ParetoWs carve_pareto(void *ws, int64_t m) {
  ParetoWs w;
  unsigned char *p = reinterpret_cast<unsigned char *>(ws);
  const int64_t mb = round_up(m, 256);
  w.flags = p;                    p += mb;
  w.counts = (int32_t *)p;        p += round_up(ceil_div(m, PB) * 4 + 4, 256);
  w.listA = (int32_t *)p;         p += mb * 4;
  w.listS = (int32_t *)p;         p += round_up((int64_t)PARETO_SAMPLE * 4, 256);
  w.nS = (int32_t *)p;            p += 256;
  w.nA = (int32_t *)p;            p += 256;
  w.key = reinterpret_cast<unsigned long long *>(w.nS + 32);
  return w;
}

size_t pareto_ws_bytes(int64_t m) {
  const int64_t mb = round_up(m, 256);
  return (size_t)(mb + round_up(ceil_div(m, PB) * 4 + 4, 256) + mb * 4 + round_up((int64_t)PARETO_SAMPLE * 4, 256) + 512);
}

static void compact(const uint8_t *flags, const int32_t *idxA, const int32_t *nA_ptr, int nA_host, int strideA,
                    int32_t *counts, int32_t *out_idx, int32_t *out_count, cudaStream_t st) {
  const int nblocks = (int)ceil_div(nA_host, PB);
  compact_count_kernel<<<nblocks, PB, 0, st>>>(flags, nA_ptr, nA_host, counts);
  compact_scan_kernel<<<1, 1024, 0, st>>>(counts, nblocks, out_count);
  compact_scatter_kernel<<<nblocks, PB, 0, st>>>(flags, idxA, nA_ptr, nA_host, strideA, counts, out_idx);
}

template <int K>
static int pareto_impl(const float *F, int64_t m, int64_t ldf, const float *cv, int32_t *idx_out, int32_t *count, void *ws,
                       int64_t ws_bytes, cudaStream_t st) {
  if (m <= 0 || m > 0x7fffffff) return HB_ERR_INVALID;
  if ((size_t)ws_bytes < pareto_ws_bytes(m)) return HB_ERR_INVALID;
  ParetoWs w = carve_pareto(ws, m);
  const int mi = (int)m;
  // B-list segments per launch: enough blocks to fill the machine when list A is short
  auto segs = [](int nA, int nB) {
    const int ablocks = (int)ceil_div(nA, PB);
    int s = (int)ceil_div(592, ablocks);                       // ~4 blocks per SM
    const int smax = (int)ceil_div(nB, PB);
    return s < 1 ? 1 : (s > smax ? (smax < 1 ? 1 : smax) : s);
  };
  if (mi <= PARETO_DIRECT_MAX) {
    HB_CUDA(cudaMemsetAsync(w.flags, 1, (size_t)mi, st));
    nondominated_kernel<K><<<dim3((unsigned)ceil_div(mi, PB), (unsigned)segs(mi, mi)), PB, 0, st>>>(F, ldf, cv, nullptr, nullptr, mi, 1, nullptr, nullptr, mi, 1, w.flags);
    compact(w.flags, nullptr, nullptr, mi, 1, w.counts, idx_out, count, st);
    count_launches(4);
  } else {
    // (1) exact front of a strided sample
    const int stride = (int)(m / PARETO_SAMPLE);
    const int ns = PARETO_SAMPLE;
    HB_CUDA(cudaMemsetAsync(w.flags, 1, (size_t)ns, st));
    nondominated_kernel<K><<<dim3((unsigned)ceil_div(ns, PB), (unsigned)segs(ns, ns)), PB, 0, st>>>(F, ldf, cv, nullptr, nullptr, ns, stride, nullptr, nullptr, ns, stride, w.flags);
    compact(w.flags, nullptr, nullptr, ns, stride, w.counts, w.listS, w.nS, st);
    // (2) all points against the sample front (a short list: one segment)
    HB_CUDA(cudaMemsetAsync(w.flags, 1, (size_t)mi, st));
    nondominated_kernel<K><<<(int)ceil_div(mi, PB), PB, 0, st>>>(F, ldf, cv, nullptr, nullptr, mi, 1, w.listS, w.nS, 0, 1, w.flags);
    compact(w.flags, nullptr, nullptr, mi, 1, w.counts, w.listA, w.nA, st);
    // (3) exact all-pairs among the survivors (count known only on the device: launch for the upper bound; blocks past the
    //     count exit at once; four B segments keep a long survivor list from serialising on a few SMs)
    HB_CUDA(cudaMemsetAsync(w.flags, 1, (size_t)mi, st));
    nondominated_kernel<K><<<dim3((unsigned)ceil_div(mi, PB), 4), PB, 0, st>>>(F, ldf, cv, w.listA, w.nA, 0, 1, w.listA, w.nA, 0, 1, w.flags);
    compact(w.flags, w.listA, w.nA, mi, 1, w.counts, idx_out, count, st);
    count_launches(12);
  }
  if (cv) {
    HB_CUDA(cudaMemsetAsync(w.key, 0xff, sizeof(unsigned long long), st));
    least_cv_kernel<K><<<(int)ceil_div(mi, PB), PB, 0, st>>>(F, ldf, cv, mi, w.key);
    least_cv_apply_kernel<<<1, 1, 0, st>>>(w.key, idx_out, count);
    count_launches(2);
  }
  HB_LAUNCH_CHECK("pareto");
  return HB_OK;
}

int launch_pareto(const float *F, int64_t m, int K, int64_t ldf, const float *cv, int32_t *idx_out, int32_t *count, void *ws,
                  int64_t ws_bytes, cudaStream_t st) {
  if (ldf < K) return HB_ERR_INVALID;
  switch (K) {
    case 1: return pareto_impl<1>(F, m, ldf, cv, idx_out, count, ws, ws_bytes, st);
    case 2: return pareto_impl<2>(F, m, ldf, cv, idx_out, count, ws, ws_bytes, st);
    case 3: return pareto_impl<3>(F, m, ldf, cv, idx_out, count, ws, ws_bytes, st);
    case 4: return pareto_impl<4>(F, m, ldf, cv, idx_out, count, ws, ws_bytes, st);
    case 5: return pareto_impl<5>(F, m, ldf, cv, idx_out, count, ws, ws_bytes, st);
    case 6: return pareto_impl<6>(F, m, ldf, cv, idx_out, count, ws, ws_bytes, st);
    case 7: return pareto_impl<7>(F, m, ldf, cv, idx_out, count, ws, ws_bytes, st);
    case 8: return pareto_impl<8>(F, m, ldf, cv, idx_out, count, ws, ws_bytes, st);
    default: return HB_ERR_INVALID;
  }
}

int launch_pareto3(const float *F, int64_t m, int32_t *idx_out, int32_t *count, void *ws, int64_t ws_bytes,
                   cudaStream_t st) {
  return launch_pareto(F, m, 3, 3, nullptr, idx_out, count, ws, ws_bytes, st);
}

// ================================================================================= multi-GPU front exchange
// Fixed-capacity front buffers for the ONE all-gather of the sharded scoring path (SURVEY 8e), built and merged on the
// device so that a step needs no host synchronisation before its result is read:
//   buffer [(capacity + 1), FRONT_W] floats.  row 0 = (count, overflow flag, 0...);  row 1 + j = (F0, F1, F2, mu, sigma,
//   id_lo, id_hi, 0) of front row j, the global candidate id split in two fp32-exact 24-bit halves; unused rows = +inf.
constexpr int FRONT_W = 8;

__global__ void __launch_bounds__(256) front_pack_kernel(const float *__restrict__ F, const float *__restrict__ mu,
                                                         const float *__restrict__ var, const int32_t *__restrict__ idx,
                                                         const int32_t *__restrict__ count, int64_t row_offset, int capacity,
                                                         float *__restrict__ out) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r > capacity) return;
  const int k = *count;
  float v[FRONT_W];
  if (r == 0) {
    v[0] = (float)k;
    v[1] = k > capacity ? 1.0f : 0.0f;
#pragma unroll
    for (int u = 2; u < FRONT_W; ++u) v[u] = 0.0f;
  } else if (r - 1 < min(k, capacity)) {
    const int64_t i = idx[r - 1];
    const int64_t gid = row_offset + i;
    v[0] = F[i * 3 + 0];
    v[1] = F[i * 3 + 1];
    v[2] = F[i * 3 + 2];
    v[3] = mu ? mu[i] : 0.0f;
    v[4] = var ? sqrtf(var[i]) : 0.0f;
    v[5] = (float)(gid & 0xFFFFFF);
    v[6] = (float)(gid >> 24);
    v[7] = 0.0f;
  } else {
#pragma unroll
    for (int u = 0; u < FRONT_W; ++u) v[u] = u < 3 ? INFINITY : 0.0f;
  }
  float4 *o = reinterpret_cast<float4 *>(out + (int64_t)r * FRONT_W);
  o[0] = make_float4(v[0], v[1], v[2], v[3]);
  o[1] = make_float4(v[4], v[5], v[6], v[7]);
}

// gathered buffers [world][capacity + 1][FRONT_W] -> objective matrix [world * capacity, 3] (+inf beyond each rank's count)
__global__ void __launch_bounds__(256) front_unpack_kernel(const float *__restrict__ all, int world, int capacity,
                                                           float *__restrict__ Fm, int32_t *__restrict__ overflow) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= world * capacity) return;
  const int w = p / capacity, j = p - w * capacity;
  const float *hdr = all + (int64_t)w * (capacity + 1) * FRONT_W;
  const int k = (int)hdr[0];
  if (j == 0 && (k > capacity || hdr[1] != 0.0f)) atomicOr(overflow, 1);
  const float *row = hdr + (int64_t)(j + 1) * FRONT_W;
  const bool valid = j < min(k, capacity);
  Fm[(int64_t)p * 3 + 0] = valid ? row[0] : INFINITY;
  Fm[(int64_t)p * 3 + 1] = valid ? row[1] : INFINITY;
  Fm[(int64_t)p * 3 + 2] = valid ? row[2] : INFINITY;
}

__global__ void __launch_bounds__(256) front_gather_kernel(const float *__restrict__ all, int world, int capacity,
                                                           const int32_t *__restrict__ idx, const int32_t *__restrict__ count,
                                                           const int32_t *__restrict__ overflow, float *__restrict__ out) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  const int cap_total = world * capacity;
  if (r > cap_total) return;
  const int k = *count;
  float4 a, b;
  if (r == 0) {
    a = make_float4((float)k, *overflow ? 1.0f : 0.0f, 0.f, 0.f);
    b = make_float4(0.f, 0.f, 0.f, 0.f);
  } else if (r - 1 < k) {
    const int p = idx[r - 1];
    const int w = p / capacity, j = p - w * capacity;
    const float4 *src = reinterpret_cast<const float4 *>(all + ((int64_t)w * (capacity + 1) + j + 1) * FRONT_W);
    a = src[0];
    b = src[1];
  } else {
    a = make_float4(INFINITY, INFINITY, INFINITY, 0.f);
    b = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  float4 *o = reinterpret_cast<float4 *>(out + (int64_t)r * FRONT_W);
  o[0] = a;
  o[1] = b;
}

int launch_front_pack(const float *F, const float *mu, const float *var, const int32_t *idx, const int32_t *count,
                      int64_t row_offset, int64_t capacity, float *out, cudaStream_t st) {
  if (capacity <= 0 || capacity > 0x3fffffff) return HB_ERR_INVALID;
  front_pack_kernel<<<(int)ceil_div(capacity + 1, 256), 256, 0, st>>>(F, mu, var, idx, count, row_offset, (int)capacity, out);
  count_launches(1);
  HB_LAUNCH_CHECK("front_pack");
  return HB_OK;
}

size_t front_merge_ws_bytes(int64_t world, int64_t capacity) {
  const int64_t R = world * capacity;
  return (size_t)round_up(R * 3 * 4, 256) + (size_t)round_up(R * 4, 256) + 512 + pareto_ws_bytes(R);
}

int launch_front_merge(const float *all, int64_t world, int64_t capacity, float *out, void *ws, int64_t ws_bytes,
                       cudaStream_t st) {
  const int64_t R = world * capacity;
  if (world <= 0 || capacity <= 0 || R > 0x3fffffff) return HB_ERR_INVALID;
  if ((size_t)ws_bytes < front_merge_ws_bytes(world, capacity)) return HB_ERR_INVALID;
  unsigned char *p = reinterpret_cast<unsigned char *>(ws);
  float *Fm = reinterpret_cast<float *>(p);                 p += round_up(R * 3 * 4, 256);
  int32_t *idx = reinterpret_cast<int32_t *>(p);            p += round_up(R * 4, 256);
  int32_t *cnt = reinterpret_cast<int32_t *>(p);
  int32_t *ovf = cnt + 1;                                   p += 512;
  HB_CUDA(cudaMemsetAsync(cnt, 0, 2 * sizeof(int32_t), st));
  front_unpack_kernel<<<(int)ceil_div(R, 256), 256, 0, st>>>(all, (int)world, (int)capacity, Fm, ovf);
  count_launches(1);
  const int s = launch_pareto3(Fm, R, idx, cnt, p, (int64_t)pareto_ws_bytes(R), st);
  if (s != HB_OK) return s;
  front_gather_kernel<<<(int)ceil_div(R + 1, 256), 256, 0, st>>>(all, (int)world, (int)capacity, idx, cnt, ovf, out);
  count_launches(1);
  HB_LAUNCH_CHECK("front_merge");
  return HB_OK;
}

}  // namespace hb
