// CEM / iCEM population kernels: sampling, elite selection (radix select), refit, warm-start shift.
//
// Reference semantics (mbrl/planning/trajectory_opt.py):
//   CEMOptimizer._sample_population 110-128, _update_population_params 130-140, optimize 142-188
//   ICEMOptimizer.optimize 391-487;  util.math.truncated_normal_ util/math.py:69-92,
//   powerlaw_psd_gaussian util/math.py:318-396;  TrajectoryOptimizer.optimize 563-567.
#include <string.h>

#include "common.cuh"

namespace {

// ------------------------------------------------------------------------------------------------------
// sampling
// ------------------------------------------------------------------------------------------------------
// one element of the population (trajectory_opt.py:110-128): idx = sequence * dims + d
__device__ __forceinline__ float cem_sample_element(long long idx, int dims, float m, float dp, float lo, float hi,
                                                    const float* __restrict__ z, unsigned long long seed,
                                                    unsigned long long offset, int clipped, int seq0) {
  const int d = (int)(idx % dims);
  float zz;
  if (z) {
    zz = z[idx];
  } else {
    // N(0,1); truncated to [-2, 2] by redrawing violators (util/math.py:83-92) unless clipped_normal
    uint32_t attempt = 0;
    const int n_i = seq0 + (int)(idx / dims);  // GLOBAL sequence index: draws do not depend on the sharding
    while (true) {
      float g[4];
      philox_normal4((uint32_t)n_i, (uint32_t)(d >> 2), RNG_STREAM_CEM | attempt, (uint32_t)offset, seed, g);
      zz = g[d & 3];
      if (clipped || (zz >= -2.0f && zz <= 2.0f) || attempt >= 64) break;
      ++attempt;
    }
    if (!clipped) zz = fminf(fmaxf(zz, -2.0f), 2.0f);
  }
  float v;
  if (clipped) {  // trajectory_opt.py:116-120 (dispersion is a standard deviation)
    v = m + dp * zz;
    v = v > lo ? v : lo;
    v = v < hi ? v : hi;
  } else {        // trajectory_opt.py:122-128 (dispersion is a variance)
    const float l2 = (m - lo) / 2.0f, u2 = (hi - m) / 2.0f;
    const float mv = fminf(l2 * l2, u2 * u2);
    const float cv = fminf(mv, dp);
    v = zz * sqrtf(cv) + m;
  }
  return v;
}

__global__ void cem_sample_kernel(int n, int dims, const float* __restrict__ mu, const float* __restrict__ disp,
                                  const float* __restrict__ lb, const float* __restrict__ ub,
                                  const float* __restrict__ z, unsigned long long seed, unsigned long long offset,
                                  int clipped, float* __restrict__ pop, int seq0) {
  pdl_trigger();
  pdl_wait();  // mu / disp come from the previous refit; pop may still be read by the previous iteration's kernels
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)n * dims) return;
  const int d = (int)(idx % dims);
  pop[idx] = cem_sample_element(idx, dims, mu[d], disp[d], lb[d], ub[d], z, seed, offset, clipped, seq0);
}

// iCEM coloured noise: one thread per (sequence, action dim) synthesises the H samples of its series
__global__ void icem_sample_kernel(int n, int H, int A, float exponent, const float* __restrict__ mu,
                                   const float* __restrict__ var, const float* __restrict__ lb,
                                   const float* __restrict__ ub, const float* __restrict__ sr,
                                   const float* __restrict__ si, unsigned long long seed, unsigned long long offset,
                                   float* __restrict__ pop) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)n * A) return;
  const int ni = (int)(idx / A), ad = (int)(idx % A);
  const int K = H / 2 + 1;
  // spectrum scale s_k = f_k^(-beta/2), f_0 := f_1 (low-frequency cut-off 1/H); theoretical sigma
  float sig2 = 0.f;
  for (int k = 1; k < K; ++k) {
    float w = powf((float)k / (float)H, -exponent / 2.0f);
    if (k == K - 1) w *= (1.0f + (float)(H % 2)) / 2.0f;
    sig2 += w * w;
  }
  const float sigma = 2.0f * sqrtf(sig2) / (float)H;
  for (int t = 0; t < H; ++t) {
    float acc = 0.f;
    for (int k = 0; k < K; ++k) {
      const float s = powf((float)(k == 0 ? 1 : k) / (float)H, -exponent / 2.0f);
      float zr, zi;
      if (sr) {
        zr = sr[((size_t)ni * A + ad) * K + k];
        zi = si[((size_t)ni * A + ad) * K + k];
      } else {
        float g[4];
        philox_normal4((uint32_t)ni, (uint32_t)(ad * K + k), RNG_STREAM_ICEM, (uint32_t)offset, seed, g);
        zr = g[0];
        zi = g[1];
      }
      const float re = zr * s;
      float im = zi * s;
      const bool nyq = (H % 2 == 0) && (k == K - 1);
      if (k == 0 || nyq) im = 0.f;
      const int ph = (int)(((long long)k * t) % H);
      float sn, cs;
      sincospif(2.0f * (float)ph / (float)H, &sn, &cs);
      const float term = re * cs - im * sn;
      acc += (k == 0 || nyq) ? term : 2.0f * term;
    }
    const float y = acc / (float)H / sigma;
    const int d = t * A + ad;
    float v = fminf(y * sqrtf(var[d]) + mu[d], ub[d]);
    v = fmaxf(v, lb[d]);
    pop[((size_t)ni * H + t) * A + ad] = v;
  }
}

__global__ void icem_append_kernel(int keep, int H, int A, const float* __restrict__ elite,
                                   const long long* __restrict__ index, int shift, const float* __restrict__ mu,
                                   const float* __restrict__ var, const float* __restrict__ end_eps,
                                   unsigned long long seed, unsigned long long offset, float* __restrict__ dst) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= keep * H * A) return;
  const int j = idx / (H * A), t = (idx / A) % H, ad = idx % A;
  const long long src = index ? index[j] : j;
  float v;
  if (!shift) {
    v = elite[(src * H + t) * A + ad];
  } else if (t < H - 1) {
    v = elite[(src * H + t + 1) * A + ad];
  } else {  // trajectory_opt.py:451-459: fresh last action ~ N(mu[-1], sqrt(var[-1]))
    float e;
    if (end_eps) {
      e = end_eps[j * A + ad];
    } else {
      float g[4];
      philox_normal4((uint32_t)j, (uint32_t)(ad >> 2), RNG_STREAM_ICEM | 1u, (uint32_t)offset, seed, g);
      e = g[ad & 3];
    }
    v = mu[(H - 1) * A + ad] + sqrtf(var[(H - 1) * A + ad]) * e;
  }
  dst[idx] = v;
}

__global__ void shift_kernel(int H, int A, int replan, const float* __restrict__ best,
                             const float* __restrict__ init_row, float* __restrict__ prev) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= H * A) return;
  const int t = idx / A, ad = idx % A;
  prev[idx] = (t < H - replan) ? best[(t + replan) * A + ad] : init_row[ad];
}

// mean over particles of the per-row returns: model_env.py:190-191
__global__ void particle_mean_kernel(int N, int P, const float* __restrict__ total, float* __restrict__ returns) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  float s = 0.f;
  for (int p = 0; p < P; ++p) s += total[(size_t)n * P + p];
  returns[n] = s / (float)P;
}

// ------------------------------------------------------------------------------------------------------
// elite selection + refit: one CTA
// ------------------------------------------------------------------------------------------------------
constexpr int kSelThreads = 1024;
constexpr int kSmallN = 2048;  // populations up to this size are ranked by counting in shared memory

// Order-preserving key of a float for the radix selects.  -0.0 maps to the key of +0.0: the two compare equal, so they
// tie (lowest index first) exactly as in the counting paths and in torch.topk's comparisons.
__device__ __forceinline__ uint32_t order_key(float v) {
  uint32_t u = __float_as_uint(v);
  if (u == 0x80000000u) u = 0u;
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__device__ __forceinline__ int block_exclusive_scan(int v, int* warp_sums, int* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int n = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += n;
  }
  if (lane == 31) warp_sums[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    int w = warp_sums[lane];
    int winc = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int n = __shfl_up_sync(0xffffffffu, winc, o);
      if (lane >= o) winc += n;
    }
    warp_sums[lane] = winc - w;
    if (lane == 31) *total = winc;
  }
  __syncthreads();
  int res = warp_sums[warp] + inc - v;
  __syncthreads();
  return res;
}

struct SelArgs {
  int n, dims, k;
  float alpha;
  int unbiased, use_std;
  int mode;  // 0: refit in place, 1: emit top-k records only
  const float* pop;
  long long pstride;
  float* values;
  long long vstride;
  float* mu;
  float* disp;
  float* best_value;
  float* best_solution;
  int* elite_idx;
  float* elites_out;
  float* records;
  float* partial;  // [32][dims] scratch
};

__global__ void __launch_bounds__(kSelThreads, 1) cem_select_kernel(const SelArgs s_in) {
  extern __shared__ float sel_dyn_smem[];  // [33][dims] partial sums when they fit, else the global workspace is used
  SelArgs s = s_in;
  if (s.partial == nullptr) s.partial = sel_dyn_smem;
  __shared__ int hist[256];
  __shared__ int warp_sums[32];
  __shared__ int sh_total;
  __shared__ uint32_t sh_prefix;
  __shared__ int sh_krem;
  __shared__ float sh_bestv[32];
  __shared__ int sh_besti[32];
  const int tid = threadIdx.x;
  const int n = s.n, k = s.k;

  // NaN -> -1e-10 (trajectory_opt.py:178), in place like the reference
  for (int i = tid; i < n; i += kSelThreads) {
    float v = s.values[i * s.vstride];
    if (isnan(v)) s.values[i * s.vstride] = -1e-10f;
  }
  __syncthreads();

  float bv;
  int bi;
  if (n <= kSmallN) {
    // ---- small populations (the PETS configurations): rank by counting, everything in shared memory ----
    __shared__ float sv[kSmallN];
    __shared__ unsigned char sf[kSmallN];
    for (int i = tid; i < n; i += kSelThreads) sv[i] = s.values[i * s.vstride];
    if (tid == 0) sh_besti[0] = 0;
    __syncthreads();
    for (int i = tid; i < n; i += kSelThreads) {
      const float vi = sv[i];
      int rank = 0;
      for (int j = 0; j < n; ++j) {
        const float vj = sv[j];
        rank += (vj > vi || (vj == vi && j < i)) ? 1 : 0;
      }
      sf[i] = rank < k ? 1 : 0;
      if (rank == 0) sh_besti[0] = i;  // the maximum, lowest index on ties
    }
    __syncthreads();
    for (int i = tid; i < n; i += kSelThreads) {
      if (sf[i]) {
        int pos = 0;
        for (int j = 0; j < i; ++j) pos += sf[j];
        s.elite_idx[pos] = i;
      }
    }
    __syncthreads();
    bi = sh_besti[0];
    bv = sv[bi];
  } else {
  if (tid == 0) {
    sh_prefix = 0;
    sh_krem = k;
  }
  __syncthreads();
  // ---- radix select of the k-th largest key, most significant byte first ----
  for (int pass = 0; pass < 4; ++pass) {
    const int shift = 24 - 8 * pass;
    for (int b = tid; b < 256; b += kSelThreads) hist[b] = 0;
    __syncthreads();
    const uint32_t prefix = sh_prefix;
    const uint32_t mask = pass == 0 ? 0u : (0xFFFFFFFFu << (shift + 8));
    for (int i = tid; i < n; i += kSelThreads) {
      uint32_t key = order_key(s.values[i * s.vstride]);
      if ((key & mask) == prefix) atomicAdd(&hist[(key >> shift) & 0xFF], 1);
    }
    __syncthreads();
    if (tid == 0) {
      int krem = sh_krem, cum = 0, d = 255;
      for (; d > 0; --d) {
        if (cum + hist[d] >= krem) break;
        cum += hist[d];
      }
      sh_krem = krem - cum;
      sh_prefix = prefix | ((uint32_t)d << shift);
    }
    __syncthreads();
  }
  const uint32_t T = sh_prefix;  // key of the k-th largest value
  const int need_eq = sh_krem;   // how many elements equal to T belong to the top-k (lowest indices first)

  // ---- ordered compaction of the selected indices ----
  int base_sel = 0, base_eq = 0;
  for (int c0 = 0; c0 < n; c0 += kSelThreads) {
    const int i = c0 + tid;
    uint32_t key = i < n ? order_key(s.values[i * s.vstride]) : 0u;
    const int gt = (i < n && key > T) ? 1 : 0;
    const int eq = (i < n && key == T) ? 1 : 0;
    int tot_eq;
    const int eq_rank = block_exclusive_scan(eq, warp_sums, &sh_total);
    tot_eq = sh_total;
    const int sel = gt | (eq && (base_eq + eq_rank) < need_eq ? 1 : 0);
    const int pos = block_exclusive_scan(sel, warp_sums, &sh_total);
    const int tot_sel = sh_total;
    if (sel) s.elite_idx[base_sel + pos] = i;
    base_sel += tot_sel;
    base_eq += tot_eq;
    __syncthreads();
  }

  // ---- best value: max, lowest index on ties (best_values[0] / elite_idx[0] of topk) ----
  bv = -INFINITY;
  bi = 0x7fffffff;
  for (int i = tid; i < n; i += kSelThreads) {
    float v = s.values[i * s.vstride];
    if (v > bv || (v == bv && i < bi)) { bv = v; bi = i; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    float ov = __shfl_xor_sync(0xffffffffu, bv, o);
    int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
  }
  if ((tid & 31) == 0) { sh_bestv[tid >> 5] = bv; sh_besti[tid >> 5] = bi; }
  __syncthreads();
  if (tid < 32) {
    bv = sh_bestv[tid];
    bi = sh_besti[tid];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
    }
    if (tid == 0) { sh_bestv[0] = bv; sh_besti[0] = bi; }
  }
  __syncthreads();
  bv = sh_bestv[0];
  bi = sh_besti[0];

  }

  if (s.mode == 1) {  // records [k][1 + dims]
    for (int idx = tid; idx < k * (s.dims + 1); idx += kSelThreads) {
      const int j = idx / (s.dims + 1), c = idx % (s.dims + 1);
      const int src = s.elite_idx[j];
      s.records[idx] = c == 0 ? s.values[src * s.vstride] : s.pop[src * s.pstride + (c - 1)];
    }
    return;
  }

  // ---- mean / variance over the elites: warps split the elite list, lanes stride the coordinates ----
  const int warp = tid >> 5, lane = tid & 31;
  const int dims = s.dims;
  for (int d = lane; d < dims; d += 32) {
    float acc = 0.f;
    for (int e = warp; e < k; e += 32) acc += s.pop[s.elite_idx[e] * s.pstride + d];
    s.partial[warp * dims + d] = acc;
  }
  __syncthreads();
  for (int d = tid; d < dims; d += kSelThreads) {
    float acc = 0.f;
    for (int w = 0; w < 32; ++w) acc += s.partial[w * dims + d];
    s.partial[32 * dims + d] = acc / (float)k;  // mean
  }
  __syncthreads();
  for (int d = lane; d < dims; d += 32) {
    const float mean = s.partial[32 * dims + d];
    float acc = 0.f;
    for (int e = warp; e < k; e += 32) {
      float df = s.pop[s.elite_idx[e] * s.pstride + d] - mean;
      acc += df * df;
    }
    s.partial[warp * dims + d] = acc;
  }
  __syncthreads();
  for (int d = tid; d < dims; d += kSelThreads) {
    float acc = 0.f;
    for (int w = 0; w < 32; ++w) acc += s.partial[w * dims + d];
    const float mean = s.partial[32 * dims + d];
    float var = acc / (float)(s.unbiased ? (k - 1) : k);
    float nd = s.use_std ? sqrtf(var) : var;
    s.mu[d] = s.alpha * s.mu[d] + (1.0f - s.alpha) * mean;
    s.disp[d] = s.alpha * s.disp[d] + (1.0f - s.alpha) * nd;
  }
  if (s.elites_out) {
    // the reference keeps `population[elite_idx]` in topk order (descending value, trajectory_opt.py:475-476) and
    // iCEM indexes that order with randperm: emit rows by descending value (ties: lower population index first)
    for (int e = tid; e < k; e += kSelThreads) {
      const int ie = s.elite_idx[e];
      const float ve = s.values[ie * s.vstride];
      int rank = 0;
      for (int f = 0; f < k; ++f) {
        const float vf = s.values[s.elite_idx[f] * s.vstride];
        rank += (vf > ve || (vf == ve && f < e)) ? 1 : 0;
      }
      for (int d = 0; d < dims; ++d) s.elites_out[(size_t)rank * dims + d] = s.pop[ie * s.pstride + d];
    }
  }
  // ---- best-so-far (trajectory_opt.py:184-186) ----
  const bool better = bv > *s.best_value;
  __syncthreads();
  if (better) {
    for (int d = tid; d < dims; d += kSelThreads) s.best_solution[d] = s.pop[bi * s.pstride + d];
    if (tid == 0) *s.best_value = bv;
  }
}


// Small populations (every PETS configuration: n <= 2048) with the elite rows staged in shared memory: one CTA,
// six short phases, no global scratch.  Optionally fuses the particle mean (model_env.py:190-191) in front: values
// are then computed from the per-row totals of the rollout kernel.  Same selection rule as cem_select_kernel (NaN ->
// -1e-10, top-k by value, ties -> lowest index, elite_idx ascending); mean / variance are summed per coordinate over the
// elites in ascending index order (a fixed order: the refit is bit-identical however the population was sharded).
static __device__ __forceinline__ void select_small_body(const SelArgs& s, const float* __restrict__ row_totals, int P) {
  extern __shared__ float esm[];  // [k][dims] elite rows
  __shared__ float sv[kSmallN];
  __shared__ unsigned char sf[kSmallN];
  __shared__ int eidx[kSmallN];
  __shared__ int sh_best;
  __shared__ int sel_warp_sums[32];
  __shared__ int sel_total;
  const int tid = threadIdx.x;
  const int n = s.n, k = s.k, dims = s.dims;
  for (int i = tid; i < n; i += kSelThreads) {
    float v;
    if (row_totals) {
      float acc = 0.f;
      for (int p = 0; p < P; ++p) acc += row_totals[(size_t)i * P + p];
      v = acc / (float)P;
    } else {
      v = s.values[i * s.vstride];
    }
    const bool nan = isnan(v);
    if (nan) v = -1e-10f;  // trajectory_opt.py:178, in place like the reference
    if (nan || row_totals) s.values[i * s.vstride] = v;
    sv[i] = v;
  }
  if (tid == 0) sh_best = 0;
  __syncthreads();
  // rank by counting (vj > vi, ties -> lower index first); T threads share one candidate's n comparisons (500 sequences: 2)
  int T = 1;
  while (T < 32 && 2 * T * n <= kSelThreads) T *= 2;
  for (int base = 0; base < n; base += kSelThreads / T) {
    const int i = base + tid / T, part = tid % T;  // T divides 32: the partners of a candidate sit in one warp
    int rank = 0;
    if (i < n) {
      const float vi = sv[i];
      for (int j = part; j < n; j += T) {
        const float vj = sv[j];
        rank += (vj > vi || (vj == vi && j < i)) ? 1 : 0;
      }
    }
    for (int o = T >> 1; o > 0; o >>= 1) rank += __shfl_xor_sync(0xffffffffu, rank, o);
    if (i < n && part == 0) {
      sf[i] = rank < k ? 1 : 0;
      if (rank == 0) sh_best = i;  // the maximum, lowest index on ties
    }
  }
  __syncthreads();
  {  // ascending positions of the selected indices: block-wide exclusive scan of the flags
    int base_sel = 0;
    for (int c0 = 0; c0 < n; c0 += kSelThreads) {
      const int i = c0 + tid;
      const int flag = i < n ? (int)sf[i] : 0;
      const int pos = block_exclusive_scan(flag, sel_warp_sums, &sel_total);
      if (flag) {
        eidx[base_sel + pos] = i;
        s.elite_idx[base_sel + pos] = i;
      }
      base_sel += sel_total;
      __syncthreads();
    }
  }
  for (int idx = tid; idx < k * dims; idx += kSelThreads) {
    const int e = idx / dims, d = idx - e * dims;
    esm[idx] = s.pop[eidx[e] * s.pstride + d];
  }
  const int bi = sh_best;
  const float bv = sv[bi];
  const bool better = s.mode == 0 && bv > *s.best_value;  // read before anybody writes it
  __syncthreads();
  if (s.mode == 1) {  // records [k][1 + dims]
    for (int idx = tid; idx < k * (dims + 1); idx += kSelThreads) {
      const int j = idx / (dims + 1), c = idx - j * (dims + 1);
      s.records[idx] = c == 0 ? sv[eidx[j]] : esm[j * dims + (c - 1)];
    }
    return;
  }
  for (int d = tid; d < dims; d += kSelThreads) {
    float acc = 0.f;
    for (int e = 0; e < k; ++e) acc += esm[e * dims + d];
    const float mean = acc / (float)k;
    float acc2 = 0.f;
    for (int e = 0; e < k; ++e) {
      const float df = esm[e * dims + d] - mean;
      acc2 += df * df;
    }
    const float var = acc2 / (float)(s.unbiased ? (k - 1) : k);
    const float nd = s.use_std ? sqrtf(var) : var;
    s.mu[d] = s.alpha * s.mu[d] + (1.0f - s.alpha) * mean;
    s.disp[d] = s.alpha * s.disp[d] + (1.0f - s.alpha) * nd;
    if (better) s.best_solution[d] = s.pop[bi * s.pstride + d];
  }
  if (s.elites_out) {  // rows by descending value (ties: lower population index first), trajectory_opt.py:475-476
    for (int e = tid; e < k; e += kSelThreads) {
      const float ve = sv[eidx[e]];
      int rank = 0;
      for (int f = 0; f < k; ++f) {
        const float vf = sv[eidx[f]];
        rank += (vf > ve || (vf == ve && f < e)) ? 1 : 0;
      }
      for (int d = 0; d < dims; ++d) s.elites_out[(size_t)rank * dims + d] = esm[e * dims + d];
    }
  }
  if (better && tid == 0) *s.best_value = bv;
}

__global__ void __launch_bounds__(kSelThreads, 1)
cem_select_small_kernel(const SelArgs s, const float* __restrict__ row_totals, int P) {
  pdl_trigger();
  pdl_wait();  // values / row totals / population are the previous kernels' outputs
  select_small_body(s, row_totals, P);
}

// Refit of iteration i AND the population of iteration i + 1 in one launch (2 launches per CEM iteration: rollout, this).
// CTA 0 runs the refit above and then publishes a tag; the other CTAs of the (small, co-resident: <= 64 CTAs, CTA 0 is
// dispatched first) grid spin on it, then every CTA draws its slice of the next population from the new (mu, dispersion).
// refit = 0: sample only (the first iteration's population); sample = 0: refit only (the last iteration).
struct NextPop {
  int refit, sample;
  int n_pop;  // sequences to draw (this rank's shard); the refit may run over a different number of rows (gathered records)
  const float* lb;
  const float* ub;
  const float* z;  // injected noise of the NEXT iteration or NULL
  unsigned long long seed, offset;
  int clipped, seq0;
  unsigned int* flag;
  unsigned int tag;
  float* pop_out;
};

__global__ void __launch_bounds__(kSelThreads, 1)
cem_refit_sample_kernel(const SelArgs s, const float* __restrict__ row_totals, int P, const NextPop q) {
  pdl_trigger();
  pdl_wait();
  if (q.refit) {
    if (blockIdx.x == 0) {
      select_small_body(s, row_totals, P);
      __syncthreads();  // every read of the old population (elite rows, best row) is done
      if (threadIdx.x == 0) {
        __threadfence();
        asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(q.flag), "r"(q.tag) : "memory");
      }
    } else {
      if (threadIdx.x == 0) {
        unsigned int v;
        do {
          asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(q.flag) : "memory");
        } while (v != q.tag);
      }
      __syncthreads();
    }
  }
  if (!q.sample) return;
  const long long tot = (long long)q.n_pop * s.dims;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < tot; idx += (long long)gridDim.x * blockDim.x) {
    const int d = (int)(idx % s.dims);
    q.pop_out[idx] = cem_sample_element(idx, s.dims, __ldcg(s.mu + d), __ldcg(s.disp + d), q.lb[d], q.ub[d], q.z, q.seed, q.offset,
                                        q.clipped, q.seq0);
  }
}

// ------------------------------------------------------------------------------------------------------
// MPPI (mbrl/planning/trajectory_opt.py:191-311)
// ------------------------------------------------------------------------------------------------------
// beta-smoothed noisy actions, sequential over the horizon (trajectory_opt.py:262-287): one thread per (n, action dim).
// NB the reference overwrites the variance-scaled population with mean + *unscaled* truncated noise; restated as is.
__global__ void mppi_sample_kernel(int n, int H, int A, float beta, const float* __restrict__ mean,
                                   const float* __restrict__ past, const float* __restrict__ lb,
                                   const float* __restrict__ ub, const float* __restrict__ z, unsigned long long seed,
                                   unsigned long long offset, float* __restrict__ pop) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)n * A) return;
  const int ni = (int)(idx / A), ad = (int)(idx % A);
  float prev = past[ad];
  for (int t = 0; t < H; ++t) {
    const int d = t * A + ad;
    float zz;
    if (z) {
      zz = z[((size_t)ni * H + t) * A + ad];
    } else {
      uint32_t attempt = 0;
      while (true) {
        float g[4];
        philox_normal4((uint32_t)ni, (uint32_t)(d >> 2), RNG_STREAM_CEM | attempt, (uint32_t)offset, seed, g);
        zz = g[d & 3];
        if ((zz >= -2.0f && zz <= 2.0f) || attempt >= 64) break;
        ++attempt;
      }
      zz = fminf(fmaxf(zz, -2.0f), 2.0f);
    }
    const float v = beta * (mean[d] + zz) + (1.0f - beta) * prev;
    prev = v;  // the recurrence runs on the un-clipped value (clipping happens after the loop in the reference)
    float c = v > ub[d] ? ub[d] : v;
    c = c < lb[d] ? lb[d] : c;
    pop[((size_t)ni * H + t) * A + ad] = c;
  }
}

// softmax-weighted mean of the population (trajectory_opt.py:296-309): one CTA
__global__ void __launch_bounds__(kSelThreads, 1)
mppi_update_kernel(int n, int dims, float gamma, const float* __restrict__ pop, float* __restrict__ values,
                   float* __restrict__ mean_out, float* __restrict__ wts, float* __restrict__ partial) {
  __shared__ float red[32];
  __shared__ float sh_max, sh_norm;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float vmax = -INFINITY;
  for (int i = tid; i < n; i += kSelThreads) {
    float v = values[i];
    if (isnan(v)) { v = -1e-10f; values[i] = v; }
    vmax = fmaxf(vmax, v);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) vmax = fmaxf(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
  if (lane == 0) red[warp] = vmax;
  __syncthreads();
  if (tid < 32) {
    float v = red[tid];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    if (tid == 0) sh_max = v;
  }
  __syncthreads();
  float sum = 0.f;
  for (int i = tid; i < n; i += kSelThreads) {
    const float w = expf(gamma * (values[i] - sh_max));
    wts[i] = w;
    sum += w;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  __syncthreads();
  if (lane == 0) red[warp] = sum;
  __syncthreads();
  if (tid < 32) {
    float v = red[tid];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (tid == 0) sh_norm = v + 1e-10f;
  }
  __syncthreads();
  for (int d = lane; d < dims; d += 32) {
    float acc = 0.f;
    for (int i = warp; i < n; i += 32) acc += pop[(size_t)i * dims + d] * wts[i];
    partial[warp * dims + d] = acc;
  }
  __syncthreads();
  for (int d = tid; d < dims; d += kSelThreads) {
    float acc = 0.f;
    for (int w = 0; w < 32; ++w) acc += partial[w * dims + d];
    mean_out[d] = acc / sh_norm;
  }
}


// ------------------------------------------------------------------------------------------------------
// Sharded population: the exchange of an iteration over NVLink peer memory, fused into the select / refit kernels (no
// host-issued collective between them), and sized by the ELITE SET, not by rank count x elites:
//   cem_values_push_kernel         NaN rule on this rank's values, then the values into slot `rank` of EVERY rank's value
//                                  table (plain stores through the IPC mapping of the peer's buffer), system fence, epoch flag;
//   cem_elites_refit_sample_kernel CTA 0: waits for all value flags -> every rank now holds all N values in global index order
//                                  and runs the SAME radix select (k-th largest key, ties by lowest index) -> the rows of the
//                                  elites that live on this rank go, with their values, to their position (ascending global
//                                  index) in every rank's elite table -> epoch flag -> waits for all elite flags -> refit
//                                  (mean / unbiased variance summed in ascending index order: the single-GPU arithmetic,
//                                  bit for bit), best-so-far, tag; then every CTA draws this rank's next population shard.
// Per rank and iteration: N * 4 B of values + (1 + dims) * 4 B per elite it owns, to each peer -- where gathering "the
// local top-k of every rank" moves world x min(k, N / world) records and makes every rank select among them (at 8 ranks x
// 500 sequences, k = 400: 3 200 records of 724 B and a second select, the limiter of weak scaling in round 2's first runs).
// Two parities per table: a rank can be at most one iteration ahead of the slowest one.  Spins are bounded (~2 s) and
// report through `status`.
// ------------------------------------------------------------------------------------------------------
constexpr int kMaxPeers = 16;
struct PeerArgs {
  int rank, world, n_loc, dims, elite_num, parity;
  unsigned int epoch;
  unsigned char* base[kMaxPeers];  // this process's mapping of rank p's buffer
};

__host__ __device__ inline size_t peer_al(size_t x) { return (x + 255) & ~(size_t)255; }
__host__ __device__ inline size_t peer_vals_bytes(int world, int n_loc) { return peer_al((size_t)world * n_loc * 4); }
__host__ __device__ inline size_t peer_elite_bytes(int elite_num, int dims) { return peer_al((size_t)elite_num * (dims + 1) * 4); }
__device__ __forceinline__ float* peer_vals(const PeerArgs& a, int p) {
  return reinterpret_cast<float*>(a.base[p] + (size_t)a.parity * peer_vals_bytes(a.world, a.n_loc));
}
__device__ __forceinline__ float* peer_elites(const PeerArgs& a, int p) {
  return reinterpret_cast<float*>(a.base[p] + 2 * peer_vals_bytes(a.world, a.n_loc) + (size_t)a.parity * peer_elite_bytes(a.elite_num, a.dims));
}
__device__ __forceinline__ unsigned int* peer_flags(const PeerArgs& a, int p, int phase) {  // [phase][parity][world]
  return reinterpret_cast<unsigned int*>(a.base[p] + 2 * peer_vals_bytes(a.world, a.n_loc) + 2 * peer_elite_bytes(a.elite_num, a.dims)) +
         ((size_t)phase * 2 + a.parity) * a.world;
}
__device__ __forceinline__ int* peer_status(const PeerArgs& a) {
  return reinterpret_cast<int*>(reinterpret_cast<unsigned int*>(a.base[a.rank] + 2 * peer_vals_bytes(a.world, a.n_loc) +
                                                                2 * peer_elite_bytes(a.elite_num, a.dims)) + 4 * a.world);
}
__device__ __forceinline__ void peer_signal(const PeerArgs& a, int phase) {  // after a system fence + barrier: threads 0..world-1
  if (threadIdx.x < a.world) {
    unsigned int* f = peer_flags(a, threadIdx.x, phase) + a.rank;
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(f), "r"(a.epoch) : "memory");
  }
}
__device__ __forceinline__ void peer_wait(const PeerArgs& a, int phase) {  // threads 0..world-1 spin, then a barrier
  if (threadIdx.x < a.world) {
    const unsigned int* f = peer_flags(a, a.rank, phase) + threadIdx.x;
    unsigned int v;
    const long long t0 = clock64();
    do {
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
      if (v != a.epoch && clock64() - t0 > 4000000000ll) {  // ~2 s: a peer never arrived
        *peer_status(a) = 1 + phase * 100 + threadIdx.x;
        break;
      }
    } while (v != a.epoch);
  }
  __syncthreads();
}

__global__ void __launch_bounds__(kSelThreads, 1) cem_values_push_kernel(float* __restrict__ values, const PeerArgs a) {
  pdl_trigger();
  pdl_wait();
  for (int i = threadIdx.x; i < a.n_loc; i += kSelThreads) {
    float v = values[i];
    if (isnan(v)) {  // trajectory_opt.py:178, in place like the reference
      v = -1e-10f;
      values[i] = v;
    }
    for (int p = 0; p < a.world; ++p) peer_vals(a, p)[(size_t)a.rank * a.n_loc + i] = v;
  }
  __threadfence_system();
  __syncthreads();
  peer_signal(a, 0);
}

struct RefitArgs {
  float alpha;
  int use_std;
  const float* pop;  // this rank's shard [n_loc][dims]
  float *mu, *disp, *best_value, *best_solution;
};

__global__ void __launch_bounds__(kSelThreads, 1)
cem_elites_refit_sample_kernel(const PeerArgs a, const RefitArgs r, const NextPop q) {
  extern __shared__ int my_pos[];  // [n_loc] position of my sequence in the ordered elite table, -1 if not an elite
  __shared__ int hist[256];
  __shared__ int warp_sums[32];
  __shared__ int sh_total;
  __shared__ uint32_t sh_prefix;
  __shared__ int sh_krem;
  __shared__ float sh_bv[32];
  __shared__ int sh_bi[32];
  pdl_trigger();
  pdl_wait();
  const int tid = threadIdx.x, dims = a.dims, k = a.elite_num;
  if (blockIdx.x == 0) {
    const int n = a.world * a.n_loc;
    peer_wait(a, 0);
    const float* vals = peer_vals(a, a.rank);
    if (tid == 0) {
      sh_prefix = 0;
      sh_krem = k;
    }
    for (int i = tid; i < a.n_loc; i += kSelThreads) my_pos[i] = -1;
    __syncthreads();
    // ---- radix select of the k-th largest key, most significant byte first (as cem_select_kernel) ----
    for (int pass = 0; pass < 4; ++pass) {
      const int shift = 24 - 8 * pass;
      for (int b = tid; b < 256; b += kSelThreads) hist[b] = 0;
      __syncthreads();
      const uint32_t prefix = sh_prefix;
      const uint32_t mask = pass == 0 ? 0u : (0xFFFFFFFFu << (shift + 8));
      for (int i = tid; i < n; i += kSelThreads) {
        const uint32_t key = order_key(__ldcg(vals + i));
        if ((key & mask) == prefix) atomicAdd(&hist[(key >> shift) & 0xFF], 1);
      }
      __syncthreads();
      if (tid == 0) {
        int krem = sh_krem, cum = 0, d = 255;
        for (; d > 0; --d) {
          if (cum + hist[d] >= krem) break;
          cum += hist[d];
        }
        sh_krem = krem - cum;
        sh_prefix = prefix | ((uint32_t)d << shift);
      }
      __syncthreads();
    }
    const uint32_t T = sh_prefix;
    const int need_eq = sh_krem;
    // ---- ordered positions (ascending global index); mine go into my_pos ----
    const int lo = a.rank * a.n_loc, hi = lo + a.n_loc;
    int base_sel = 0, base_eq = 0;
    for (int c0 = 0; c0 < n; c0 += kSelThreads) {
      const int i = c0 + tid;
      const uint32_t key = i < n ? order_key(__ldcg(vals + i)) : 0u;
      const int gt = (i < n && key > T) ? 1 : 0;
      const int eq = (i < n && key == T) ? 1 : 0;
      const int eq_rank = block_exclusive_scan(eq, warp_sums, &sh_total);
      const int tot_eq = sh_total;
      const int sel = gt | ((eq && (base_eq + eq_rank) < need_eq) ? 1 : 0);
      const int pos = block_exclusive_scan(sel, warp_sums, &sh_total);
      const int tot_sel = sh_total;
      if (sel && i >= lo && i < hi) my_pos[i - lo] = base_sel + pos;
      base_sel += tot_sel;
      base_eq += tot_eq;
      __syncthreads();
    }
    // ---- my elites -> their row of every rank's elite table: [value, sequence] ----
    const int lane = tid & 31, warp = tid >> 5;
    for (int e = warp; e < a.n_loc; e += kSelThreads / 32) {
      const int pos = my_pos[e];
      if (pos < 0) continue;
      const float v = __ldcg(vals + lo + e);
      for (int p = 0; p < a.world; ++p) {
        float* row = peer_elites(a, p) + (size_t)pos * (dims + 1);
        if (lane == 0) row[0] = v;
        for (int d = lane; d < dims; d += 32) row[1 + d] = r.pop[(size_t)e * dims + d];
      }
    }
    __threadfence_system();
    __syncthreads();
    peer_signal(a, 1);
    peer_wait(a, 1);
    // ---- refit from the k ordered elite rows: the arithmetic of select_small_body ----
    const float* el = peer_elites(a, a.rank);
    float bv = -INFINITY;
    int bi = 0x7fffffff;
    for (int e = tid; e < k; e += kSelThreads) {
      const float v = __ldcg(el + (size_t)e * (dims + 1));
      if (v > bv || (v == bv && e < bi)) { bv = v; bi = e; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
    }
    if (lane == 0) { sh_bv[warp] = bv; sh_bi[warp] = bi; }
    __syncthreads();
    bv = sh_bv[0]; bi = sh_bi[0];
    for (int w = 1; w < kSelThreads / 32; ++w)
      if (sh_bv[w] > bv || (sh_bv[w] == bv && sh_bi[w] < bi)) { bv = sh_bv[w]; bi = sh_bi[w]; }
    const bool better = bv > *r.best_value;  // read before anybody writes it
    __syncthreads();
    for (int d = tid; d < dims; d += kSelThreads) {
      float acc = 0.f;
      for (int e = 0; e < k; ++e) acc += __ldcg(el + (size_t)e * (dims + 1) + 1 + d);
      const float mean = acc / (float)k;
      float acc2 = 0.f;
      for (int e = 0; e < k; ++e) {
        const float df = __ldcg(el + (size_t)e * (dims + 1) + 1 + d) - mean;
        acc2 += df * df;
      }
      const float var = acc2 / (float)(k - 1);
      const float nd = r.use_std ? sqrtf(var) : var;
      r.mu[d] = r.alpha * r.mu[d] + (1.0f - r.alpha) * mean;
      r.disp[d] = r.alpha * r.disp[d] + (1.0f - r.alpha) * nd;
      if (better) r.best_solution[d] = __ldcg(el + (size_t)bi * (dims + 1) + 1 + d);
    }
    __syncthreads();
    if (tid == 0) {
      if (better) *r.best_value = bv;
      __threadfence();
      asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(q.flag), "r"(q.tag) : "memory");
    }
    __syncthreads();
  } else {
    if (tid == 0) {
      unsigned int v;
      const long long t0 = clock64();
      do {
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(q.flag) : "memory");
      } while (v != q.tag && clock64() - t0 < 10000000000ll);
    }
    __syncthreads();
  }
  if (!q.sample) return;
  const long long tot = (long long)q.n_pop * dims;
  for (long long idx = (long long)blockIdx.x * blockDim.x + tid; idx < tot; idx += (long long)gridDim.x * blockDim.x) {
    const int d = (int)(idx % dims);
    q.pop_out[idx] = cem_sample_element(idx, dims, __ldcg(r.mu + d), __ldcg(r.disp + d), q.lb[d], q.ub[d], q.z, q.seed, q.offset,
                                        q.clipped, q.seq0);
  }
}

}  // namespace

// ------------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------------
int launch_particle_mean(int N, int P, const float* total, float* returns, cudaStream_t stream);

extern "C" {

int b200pets_cem_sample_shard(int32_t population, int32_t first_sequence, int32_t dims, const float* mu,
                              const float* dispersion, const float* lower, const float* upper, const float* z,
                              uint64_t seed, uint64_t offset, int32_t clipped_normal, float* population_out,
                              void* stream) {
  if (population <= 0 || dims <= 0) return b200pets_set_error(B200PETS_EINVAL, "cem_sample: empty population");
  if (first_sequence < 0) return b200pets_set_error(B200PETS_EINVAL, "cem_sample: negative first_sequence");
  long long tot = (long long)population * dims;
  CUDA_TRY(launch_pdl(cem_sample_kernel, dim3((unsigned)((tot + 255) / 256)), dim3(256), 0, (cudaStream_t)stream, population,
                      dims, mu, dispersion, lower, upper, z, (unsigned long long)rng_key(seed, offset),
                      (unsigned long long)offset, (int)clipped_normal, population_out, (int)first_sequence));
  return B200PETS_OK;
}

int b200pets_cem_sample(int32_t population, int32_t dims, const float* mu, const float* dispersion,
                        const float* lower, const float* upper, const float* z, uint64_t seed, uint64_t offset,
                        int32_t clipped_normal, float* population_out, void* stream) {
  return b200pets_cem_sample_shard(population, 0, dims, mu, dispersion, lower, upper, z, seed, offset, clipped_normal,
                                   population_out, stream);
}

size_t b200pets_cem_update_workspace_bytes(int32_t population, int32_t dims, int32_t elite_num) {
  (void)population;
  return (size_t)33 * dims * sizeof(float) + (size_t)elite_num * sizeof(int32_t) + 256;
}

static int run_select(int mode, int n, int dims, int k, float alpha, int unbiased, int use_std, const float* pop,
                      long long pstride, float* values, long long vstride, float* mu, float* disp, float* best_value,
                      float* best_solution, int32_t* elite_idx, float* elites_out, float* records, void* workspace,
                      size_t workspace_bytes, void* stream, const float* row_totals = nullptr, int particles = 1) {
  if (n <= 0 || dims <= 0 || k <= 0 || k > n)
    return b200pets_set_error(B200PETS_EINVAL, "cem_update: need 0 < elite_num (%d) <= population (%d)", k, n);
  if (mode == 0 && unbiased && k < 2)
    return b200pets_set_error(B200PETS_EINVAL, "cem_update: unbiased variance needs at least 2 elites");
  size_t need = b200pets_cem_update_workspace_bytes(n, dims, k);
  if (workspace_bytes < need) return b200pets_set_error(B200PETS_EINVAL, "cem_update: workspace too small (%zu < %zu)", workspace_bytes, need);
  SelArgs s{};
  s.n = n; s.dims = dims; s.k = k; s.alpha = alpha; s.unbiased = unbiased; s.use_std = use_std; s.mode = mode;
  s.pop = pop; s.pstride = pstride; s.values = values; s.vstride = vstride; s.mu = mu; s.disp = disp;
  s.best_value = best_value; s.best_solution = best_solution; s.elites_out = elites_out; s.records = records;
  s.partial = reinterpret_cast<float*>(workspace);
  s.elite_idx = elite_idx ? elite_idx : reinterpret_cast<int*>(reinterpret_cast<float*>(workspace) + 33 * (size_t)dims);
  if (n <= kSmallN && (size_t)k * dims * sizeof(float) <= 150 * 1024) {  // the PETS configurations: elites in smem
    const size_t esm = (size_t)k * dims * sizeof(float);
    CUDA_TRY(cudaFuncSetAttribute(cem_select_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 150 * 1024));
    CUDA_TRY(launch_pdl(cem_select_small_kernel, dim3(1), dim3(kSelThreads), esm, (cudaStream_t)stream, s, row_totals, particles));
    return B200PETS_OK;
  }
  if (row_totals) {  // large populations: particle mean as its own (multi-CTA) kernel, then the radix-select path
    if (vstride != 1) return b200pets_set_error(B200PETS_EINVAL, "cem_update: row totals need contiguous values");
    int rcm = launch_particle_mean(n, particles, row_totals, values, (cudaStream_t)stream);
    if (rcm) return rcm;
  }
  size_t dyn = 0;
  if ((size_t)33 * dims * sizeof(float) <= 160 * 1024) {  // partial sums in shared memory (latency-bound reduction)
    dyn = (size_t)33 * dims * sizeof(float);
    s.partial = nullptr;
    // the attribute is per device: set it on every call (cheap) rather than caching it per process
    CUDA_TRY(cudaFuncSetAttribute(cem_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
  }
  cem_select_kernel<<<1, kSelThreads, dyn, (cudaStream_t)stream>>>(s);
  CUDA_TRY(cudaGetLastError());
  return B200PETS_OK;
}

int b200pets_cem_update(int32_t population, int32_t dims, int32_t elite_num, float alpha, int32_t unbiased,
                        int32_t use_std, const float* population_in, float* values, float* mu, float* dispersion,
                        float* best_value, float* best_solution, int32_t* elite_idx, float* elites_out,
                        void* workspace, size_t workspace_bytes, void* stream) {
  return run_select(0, population, dims, elite_num, alpha, unbiased, use_std, population_in, dims, values, 1, mu,
                    dispersion, best_value, best_solution, elite_idx, elites_out, nullptr, workspace, workspace_bytes,
                    stream);
}

int b200pets_cem_local_topk(int32_t population, int32_t dims, int32_t k, const float* population_in, float* values,
                            float* records, void* workspace, size_t workspace_bytes, void* stream) {
  return run_select(1, population, dims, k, 0.f, 0, 0, population_in, dims, values, 1, nullptr, nullptr, nullptr,
                    nullptr, nullptr, nullptr, records, workspace, workspace_bytes, stream);
}

int b200pets_cem_update_from_records(int32_t num_records, int32_t dims, int32_t elite_num, float alpha,
                                     int32_t unbiased, int32_t use_std, float* records, float* mu, float* dispersion,
                                     float* best_value, float* best_solution, float* elites_out, void* workspace,
                                     size_t workspace_bytes, void* stream) {
  return run_select(0, num_records, dims, elite_num, alpha, unbiased, use_std, records + 1, dims + 1, records,
                    dims + 1, mu, dispersion, best_value, best_solution, nullptr, elites_out, nullptr, workspace,
                    workspace_bytes, stream);
}

// ---- peer-memory exchange of the sharded CEM (see cem_values_push_kernel) -----------------------------------------------
size_t b200pets_peer_buffer_bytes(int32_t world, int32_t local_population, int32_t dims, int32_t elite_num) {
  if (world <= 0 || local_population <= 0 || dims <= 0 || elite_num <= 0) return 0;
  return 2 * peer_vals_bytes(world, local_population) + 2 * peer_elite_bytes(elite_num, dims) + peer_al((size_t)(4 * world + 1) * 4);
}

int b200pets_peer_alloc(size_t bytes, void** ptr, uint8_t* ipc_handle64) {
  if (!ptr || !ipc_handle64 || bytes == 0) return b200pets_set_error(B200PETS_EINVAL, "peer_alloc: null argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  CUDA_TRY(cudaMalloc(ptr, bytes));
  CUDA_TRY(cudaMemset(*ptr, 0, bytes));
  CUDA_TRY(cudaDeviceSynchronize());
  cudaIpcMemHandle_t h;
  CUDA_TRY(cudaIpcGetMemHandle(&h, *ptr));
  memcpy(ipc_handle64, &h, 64);
  return B200PETS_OK;
}

int b200pets_peer_open(const uint8_t* ipc_handle64, void** ptr) {
  if (!ptr || !ipc_handle64) return b200pets_set_error(B200PETS_EINVAL, "peer_open: null argument");
  cudaIpcMemHandle_t h;
  memcpy(&h, ipc_handle64, 64);
  CUDA_TRY(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return B200PETS_OK;
}

int b200pets_peer_close(void* ptr, int32_t owned) {
  if (!ptr) return B200PETS_OK;
  if (owned) CUDA_TRY(cudaFree(ptr));
  else CUDA_TRY(cudaIpcCloseMemHandle(ptr));
  return B200PETS_OK;
}

static int fill_peer_args(PeerArgs* a, int rank, int world, int n_loc, int dims, int elite_num, unsigned int epoch, void* const* peer_bufs) {
  if (world < 1 || world > kMaxPeers || rank < 0 || rank >= world || !peer_bufs)
    return b200pets_set_error(B200PETS_EINVAL, "peer exchange: need 1 <= world <= %d and the peers' buffers", kMaxPeers);
  if (n_loc <= 0 || dims <= 0 || elite_num < 2 || elite_num > world * n_loc || epoch == 0)
    return b200pets_set_error(B200PETS_EINVAL, "peer exchange: need 2 <= elite_num (%d) <= population (%d) and epoch > 0", elite_num, world * n_loc);
  a->rank = rank; a->world = world; a->n_loc = n_loc; a->dims = dims; a->elite_num = elite_num;
  a->epoch = epoch; a->parity = (int)(epoch & 1u);
  for (int p = 0; p < world; ++p) {
    if (!peer_bufs[p]) return b200pets_set_error(B200PETS_EINVAL, "peer exchange: buffer of rank %d missing", p);
    a->base[p] = reinterpret_cast<unsigned char*>(peer_bufs[p]);
  }
  return B200PETS_OK;
}

int b200pets_cem_values_push(int32_t local_population, int32_t dims, int32_t elite_num, float* values, int32_t rank,
                             int32_t world, uint32_t epoch, void* const* peer_bufs, void* stream) {
  if (!values) return b200pets_set_error(B200PETS_EINVAL, "values_push: null argument");
  PeerArgs a{};
  int rc = fill_peer_args(&a, rank, world, local_population, dims, elite_num, epoch, peer_bufs);
  if (rc) return rc;
  CUDA_TRY(launch_pdl(cem_values_push_kernel, dim3(1), dim3(kSelThreads), 0, (cudaStream_t)stream, values, a));
  return B200PETS_OK;
}

int b200pets_cem_elites_refit(int32_t local_population, int32_t first_sequence, int32_t dims, int32_t elite_num, float alpha,
                              int32_t use_std, int32_t rank, int32_t world, uint32_t epoch, void* const* peer_bufs,
                              const float* population_in, float* mu, float* dispersion, float* best_value,
                              float* best_solution, int32_t sample_next, const float* lower, const float* upper,
                              uint64_t seed, uint64_t offset, int32_t clipped_normal, uint32_t* tag_word,
                              float* population_out, void* stream) {
  if (!population_in || !mu || !dispersion || !best_value || !best_solution || !tag_word)
    return b200pets_set_error(B200PETS_EINVAL, "elites_refit: null argument");
  PeerArgs a{};
  int rc = fill_peer_args(&a, rank, world, local_population, dims, elite_num, epoch, peer_bufs);
  if (rc) return rc;
  const size_t smem = (size_t)local_population * sizeof(int);
  if (smem > 160 * 1024) return b200pets_set_error(B200PETS_EUNSUPPORTED, "elites_refit: more than 40 960 sequences per rank");
  RefitArgs r{alpha, use_std, population_in, mu, dispersion, best_value, best_solution};
  NextPop q{};
  q.refit = 1; q.sample = sample_next; q.n_pop = local_population; q.lb = lower; q.ub = upper; q.z = nullptr;
  q.seed = rng_key(seed, offset); q.offset = offset; q.clipped = clipped_normal; q.seq0 = first_sequence;
  q.flag = tag_word; q.tag = epoch; q.pop_out = population_out;
  const long long tot = (long long)local_population * dims;
  unsigned grid = sample_next ? (unsigned)min((long long)64, (tot + kSelThreads - 1) / kSelThreads) : 1u;
  if (grid < 1) grid = 1;
  CUDA_TRY(cudaFuncSetAttribute(cem_elites_refit_sample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
  CUDA_TRY(launch_pdl(cem_elites_refit_sample_kernel, dim3(grid), dim3(kSelThreads), smem, (cudaStream_t)stream, a, r, q));
  return B200PETS_OK;
}

int b200pets_icem_sample(int32_t n, int32_t horizon, int32_t act_dim, float exponent, const float* mu,
                         const float* var, const float* lower, const float* upper, const float* sr, const float* si,
                         uint64_t seed, uint64_t offset, float* population_out, void* stream) {
  if (n <= 0 || horizon <= 0 || act_dim <= 0) return b200pets_set_error(B200PETS_EINVAL, "icem_sample: empty population");
  if ((sr == nullptr) != (si == nullptr)) return b200pets_set_error(B200PETS_EINVAL, "icem_sample: sr and si go together");
  long long tot = (long long)n * act_dim;
  icem_sample_kernel<<<(unsigned)((tot + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
      n, horizon, act_dim, exponent, mu, var, lower, upper, sr, si, rng_key(seed, offset), offset, population_out);
  CUDA_TRY(cudaGetLastError());
  return B200PETS_OK;
}

int b200pets_icem_append_elites(int32_t keep, int32_t horizon, int32_t act_dim, const float* elite,
                                const int64_t* index, int32_t shift, const float* mu, const float* var,
                                const float* end_eps, uint64_t seed, uint64_t offset, float* dst, void* stream) {
  if (keep <= 0) return B200PETS_OK;
  int tot = keep * horizon * act_dim;
  icem_append_kernel<<<(tot + 255) / 256, 256, 0, (cudaStream_t)stream>>>(
      keep, horizon, act_dim, elite, reinterpret_cast<const long long*>(index), shift, mu, var, end_eps, rng_key(seed, offset), offset, dst);
  CUDA_TRY(cudaGetLastError());
  return B200PETS_OK;
}


int b200pets_mppi_sample(int32_t population, int32_t horizon, int32_t act_dim, float beta, const float* mean,
                         const float* past_action, const float* lower, const float* upper, const float* z,
                         uint64_t seed, uint64_t offset, float* population_out, void* stream) {
  if (population <= 0 || horizon <= 0 || act_dim <= 0) return b200pets_set_error(B200PETS_EINVAL, "mppi_sample: empty population");
  long long tot = (long long)population * act_dim;
  mppi_sample_kernel<<<(unsigned)((tot + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
      population, horizon, act_dim, beta, mean, past_action, lower, upper, z, rng_key(seed, offset), offset, population_out);
  CUDA_TRY(cudaGetLastError());
  return B200PETS_OK;
}

size_t b200pets_mppi_update_workspace_bytes(int32_t population, int32_t dims) {
  return ((size_t)population + (size_t)32 * dims) * sizeof(float) + 256;
}

int b200pets_mppi_update(int32_t population, int32_t dims, float gamma, const float* population_in, float* values,
                         float* mean_out, void* workspace, size_t workspace_bytes, void* stream) {
  if (population <= 0 || dims <= 0) return b200pets_set_error(B200PETS_EINVAL, "mppi_update: empty population");
  if (workspace_bytes < b200pets_mppi_update_workspace_bytes(population, dims))
    return b200pets_set_error(B200PETS_EINVAL, "mppi_update: workspace too small");
  float* wts = reinterpret_cast<float*>(workspace);
  mppi_update_kernel<<<1, kSelThreads, 0, (cudaStream_t)stream>>>(population, dims, gamma, population_in, values, mean_out,
                                                                  wts, wts + population);
  CUDA_TRY(cudaGetLastError());
  return B200PETS_OK;
}

int b200pets_shift_solution(int32_t horizon, int32_t act_dim, int32_t replan_freq, const float* best,
                            const float* initial_row, float* previous_solution, void* stream) {
  if (replan_freq < 0 || replan_freq > horizon) return b200pets_set_error(B200PETS_EINVAL, "shift: replan_freq out of range");
  int tot = horizon * act_dim;
  shift_kernel<<<(tot + 255) / 256, 256, 0, (cudaStream_t)stream>>>(horizon, act_dim, replan_freq, best, initial_row,
                                                                    previous_solution);
  CUDA_TRY(cudaGetLastError());
  return B200PETS_OK;
}

}  // extern "C"

// internal (api.cu, fused plan): refit straight from the rollout kernel's per-row totals [N][P] (particle mean fused)
int launch_cem_update_rows(int population, int dims, int elite_num, float alpha, int unbiased, int use_std,
                           const float* population_in, const float* row_totals, int particles, float* values, float* mu,
                           float* dispersion, float* best_value, float* best_solution, void* workspace,
                           size_t workspace_bytes, void* stream) {
  return run_select(0, population, dims, elite_num, alpha, unbiased, use_std, population_in, dims, values, 1, mu,
                    dispersion, best_value, best_solution, nullptr, nullptr, nullptr, workspace, workspace_bytes, stream,
                    row_totals, particles);
}


bool cem_refit_sample_supported(int population, int dims, int elite_num) {
  return population <= kSmallN && (size_t)elite_num * dims * sizeof(float) <= 150 * 1024 && elite_num >= 2 && elite_num <= population;
}

// refit (particle mean fused, rows = per-particle totals) + next population; returns B200PETS_EUNSUPPORTED when the population
// is outside the single-CTA refit (the caller then uses the separate kernels)
int launch_cem_refit_sample(int population, int dims, int elite_num, float alpha, int use_std, const float* row_totals,
                            int particles, float* values, float* mu, float* dispersion, float* best_value, float* best_solution,
                            void* workspace, size_t workspace_bytes, int refit, int sample, const float* lb, const float* ub,
                            const float* z_next, unsigned long long seed, unsigned long long offset, int clipped, int seq0,
                            unsigned int* flag, unsigned int tag, float* pop, void* stream) {
  const int n = population, k = elite_num;
  if (!(n <= kSmallN && (size_t)k * dims * sizeof(float) <= 150 * 1024)) return B200PETS_EUNSUPPORTED;
  if (refit && (k < 2 || k > n)) return b200pets_set_error(B200PETS_EINVAL, "cem_update: need 2 <= elite_num (%d) <= population (%d)", k, n);
  if (workspace_bytes < b200pets_cem_update_workspace_bytes(n, dims, k)) return b200pets_set_error(B200PETS_EINVAL, "cem_update: workspace too small");
  SelArgs s{};
  s.n = n; s.dims = dims; s.k = k; s.alpha = alpha; s.unbiased = 1; s.use_std = use_std; s.mode = 0;
  s.pop = pop; s.pstride = dims; s.values = values; s.vstride = 1; s.mu = mu; s.disp = dispersion;
  s.best_value = best_value; s.best_solution = best_solution;
  s.partial = reinterpret_cast<float*>(workspace);
  s.elite_idx = reinterpret_cast<int*>(reinterpret_cast<float*>(workspace) + 33 * (size_t)dims);
  NextPop q{};
  q.refit = refit; q.sample = sample; q.n_pop = n; q.lb = lb; q.ub = ub; q.z = z_next; q.seed = seed; q.offset = offset;
  q.clipped = clipped; q.seq0 = seq0; q.flag = flag; q.tag = tag; q.pop_out = pop;
  const long long tot = (long long)n * dims;
  unsigned grid = sample ? (unsigned)min((long long)64, (tot + kSelThreads - 1) / kSelThreads) : 1u;
  if (grid < 1) grid = 1;
  const size_t esm = (size_t)k * dims * sizeof(float);
  CUDA_TRY(cudaFuncSetAttribute(cem_refit_sample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 150 * 1024));
  CUDA_TRY(launch_pdl(cem_refit_sample_kernel, dim3(grid), dim3(kSelThreads), esm, (cudaStream_t)stream, s, row_totals, particles, q));
  return B200PETS_OK;
}

int launch_particle_mean(int N, int P, const float* total, float* returns, cudaStream_t stream) {
  particle_mean_kernel<<<(N + 255) / 256, 256, 0, stream>>>(N, P, total, returns);
  CUDA_TRY(cudaGetLastError());
  return B200PETS_OK;
}
