// Particle rollout forward and the hand-written backprop-through-time.
// Reference behaviour: policy_learning/MC_PILCO.py:615-674 (apply_policy), :808-906 (4PMS variant),
// model_learning/Model_learning.py:210-229,670-718 (get_next_state), policy_learning/Policy.py:242-265,
// 323-335,389-403 (policies), policy_learning/Cost_function.py:25-36,53-182 (costs), and the autograd
// pass of MC_PILCO.py:522 which mcpilco_rollout_bwd replaces.
#include <map>
#include <utility>

#include "mcp_rollout_dev.cuh"

namespace mcp {

int gp_posterior_chunk(const McpGp& g, int E, int e, const double* Xs, int M, double* mean, double* var, double* jmean,
                       double* jvar, double* scratch, size_t scratch_doubles, cudaStream_t st);
// fused two-launches-per-step forward for small rollouts (mcp_small.cu)
bool small_path_ok(const McpRollout* r);
size_t small_path_doubles(int M, int E, int Nmax);
int rollout_fwd_small(const McpRollout* r, double* Xs, double* nv, double* scratch, size_t scratch_doubles, cudaStream_t st);
// whole-horizon persistent cluster kernel for cart-pole-sized rollouts (mcp_persist.cu)
bool persist_path_ok(const McpRollout* r);
size_t persist_path_doubles(int E);
int rollout_fwd_persist(const McpRollout* r, const double* nv0, double* scratch, size_t scratch_doubles, cudaStream_t st);
struct McpGpDev;
bool gp_posterior_batched_ok(const McpGp* gps, int E, bool jac);
size_t gp_posterior_batched_doubles(int M, int E, int nmax);
int gp_posterior_batched_setup(const McpGp* gps, int E, int M, int nmax, double* scratch, size_t scratch_doubles, const McpGpDev** tab_out,
                               double** ks_out, cudaStream_t st);
int gp_posterior_batched(const McpGpDev* tab, int E, int D, int nmax, const double* Xs, int M, double* mean, double* var, double* jmean,
                         double* jvar, double* Ks, cudaStream_t st);

// ------------------------------------------------------------------------------------------------
// forward kernels
// ------------------------------------------------------------------------------------------------
// u_t = pi(pol_in_t) with dropout and squashing, one warp per particle; then the gp-input features
// of (x_t, u_t).  Policy.py:242-265; Model_learning.py:670-683.
__global__ void __launch_bounds__(256) policy_fwd_kernel(const __grid_constant__ McpPolicy pol, const __grid_constant__ McpModel mdl,
                                                         const __grid_constant__ McpNoise nz, int M, int t, int tm,
                                                         const double* __restrict__ pol_in_t, const double* __restrict__ x_t,
                                                         double* __restrict__ u_t, double* __restrict__ Xs) {
  __shared__ double s_il[MCP_MAX_DP];
  __shared__ double s_z[8][MCP_MAX_DP];
  __shared__ double s_u[8][MCP_MAX_DU];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m = blockIdx.x * 8 + w;
  if (threadIdx.x < pol.Dp) s_il[threadIdx.x] = exp(-pol.log_ls[threadIdx.x]);
  if (m < M && lane < pol.Dp) s_z[w][lane] = policy_feature(pol, pol_in_t + (size_t)m * pol.Ds, t, lane);
  __syncthreads();
  if (m >= M) return;
  const bool drop = dropout_active(pol, nz);
  const double keep_scale = drop ? 1.0 / (1.0 - nz.p_dropout) : 1.0;
  double a[MCP_MAX_DU];
#pragma unroll
  for (int k = 0; k < MCP_MAX_DU; k++) a[k] = 0.0;
  for (int b = lane; b < pol.nb; b += 32) {
    const double* c = pol.centers + (size_t)b * pol.Dp;
    double d = 0.0;
#pragma unroll 8
    for (int j = 0; j < pol.Dp; j++) {
      double r = (s_z[w][j] - c[j]) * s_il[j];
      d = fma(r, r, d);
    }
    double h = exp(-d);
    if (drop) h = keep_unit(nz, M, pol.nb, tm, t, m, b) ? h * keep_scale : 0.0;
#pragma unroll
    for (int k = 0; k < MCP_MAX_DU; k++)
      if (k < pol.Du) a[k] = fma(pol.W[(size_t)k * pol.nb + b], h, a[k]);
  }
#pragma unroll
  for (int k = 0; k < MCP_MAX_DU; k++)
    if (k < pol.Du) {
      double v = warp_sum(a[k]);
      if (lane == 0) {
        if (pol.has_bias) v += pol.bias[k];
        if (pol.squash) v = pol.u_max[k] * tanh(v / pol.u_max[k]);
        u_t[(size_t)m * pol.Du + k] = v;
        s_u[w][k] = v;
      }
    }
  __syncwarp();
  if (Xs != nullptr && lane < mdl.D) {
    const double* x = x_t + (size_t)m * mdl.Ds;
    int j = lane;
    double f;
    if (mdl.use_trig) {
      if (j < mdl.n_na) f = x[mdl.na_idx[j]];
      else if (j < mdl.n_na + mdl.n_a) f = sin(x[mdl.a_idx[j - mdl.n_na]]);
      else if (j < mdl.n_na + 2 * mdl.n_a) f = cos(x[mdl.a_idx[j - mdl.n_na - mdl.n_a]]);
      else f = s_u[w][j - mdl.n_na - 2 * mdl.n_a];
    } else {
      f = (j < mdl.Ds) ? x[j] : s_u[w][j - mdl.Ds];
    }
    Xs[(size_t)m * mdl.D + j] = f;
  }
}

// Same policy evaluation for SMALL particle counts (the real MC-PILCO shapes, M = 200..400): one block per particle, threads over
// basis functions (up to 512 threads, so that with the reference's 200 / 400 basis functions every thread has one and the L2 round
// trips of the centre rows all overlap), so a few hundred particles still occupy every SM.
__device__ __forceinline__ void policy_block_body(const McpPolicy& pol, const McpModel& mdl, const McpNoise& nz, int M, int t, int tm,
                                                  const double* __restrict__ pol_in_t, const double* __restrict__ x_t,
                                                  double* __restrict__ u_t, double* __restrict__ Xs) {
  __shared__ double s_il[MCP_MAX_DP], s_z[MCP_MAX_DP], s_part[16][MCP_MAX_DU], s_u[MCP_MAX_DU];
  const int m = blockIdx.x, tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nw = blockDim.x >> 5;
  if (tid < pol.Dp) {
    s_il[tid] = exp(-pol.log_ls[tid]);
    s_z[tid] = policy_feature(pol, pol_in_t + (size_t)m * pol.Ds, t, tid);
  }
  __syncthreads();
  const bool drop = dropout_active(pol, nz);
  const double keep_scale = drop ? 1.0 / (1.0 - nz.p_dropout) : 1.0;
  double a[MCP_MAX_DU];
#pragma unroll
  for (int k = 0; k < MCP_MAX_DU; k++) a[k] = 0.0;
  for (int b = tid; b < pol.nb; b += blockDim.x) {
    const double* c = pol.centers + (size_t)b * pol.Dp;
    double d = 0.0;
#pragma unroll 8
    for (int j = 0; j < pol.Dp; j++) {
      double r = (s_z[j] - c[j]) * s_il[j];
      d = fma(r, r, d);
    }
    double h = exp(-d);
    if (drop) h = keep_unit(nz, M, pol.nb, tm, t, m, b) ? h * keep_scale : 0.0;
#pragma unroll
    for (int k = 0; k < MCP_MAX_DU; k++)
      if (k < pol.Du) a[k] = fma(pol.W[(size_t)k * pol.nb + b], h, a[k]);
  }
#pragma unroll
  for (int k = 0; k < MCP_MAX_DU; k++)
    if (k < pol.Du) {
      double v = warp_sum(a[k]);
      if (lane == 0) s_part[w][k] = v;
    }
  __syncthreads();
  if (tid < pol.Du) {
    double v = 0.0;
    for (int i = 0; i < nw; i++) v += s_part[i][tid];   // fixed order
    if (pol.has_bias) v += pol.bias[tid];
    if (pol.squash) v = pol.u_max[tid] * tanh(v / pol.u_max[tid]);
    u_t[(size_t)m * pol.Du + tid] = v;
    s_u[tid] = v;
  }
  __syncthreads();
  if (Xs != nullptr && tid < mdl.D) {
    const double* x = x_t + (size_t)m * mdl.Ds;
    const int j = tid;
    double f;
    if (mdl.use_trig) {
      if (j < mdl.n_na) f = x[mdl.na_idx[j]];
      else if (j < mdl.n_na + mdl.n_a) f = sin(x[mdl.a_idx[j - mdl.n_na]]);
      else if (j < mdl.n_na + 2 * mdl.n_a) f = cos(x[mdl.a_idx[j - mdl.n_na - mdl.n_a]]);
      else f = s_u[j - mdl.n_na - 2 * mdl.n_a];
    } else {
      f = (j < mdl.Ds) ? x[j] : s_u[j - mdl.Ds];
    }
    Xs[(size_t)m * mdl.D + j] = f;
  }
}

__global__ void __launch_bounds__(512) policy_fwd_block_kernel(const __grid_constant__ McpPolicy pol, const __grid_constant__ McpModel mdl,
                                                               const __grid_constant__ McpNoise nz, int M, int t, int tm,
                                                               const double* __restrict__ pol_in_t, const double* __restrict__ x_t,
                                                               double* __restrict__ u_t, double* __restrict__ Xs) {
  policy_block_body(pol, mdl, nz, M, t, tm, pol_in_t, x_t, u_t, Xs);
}

static inline int policy_block_threads(int nb) {
  const int t = (nb + 31) / 32 * 32;
  return t < 128 ? 128 : (t > 512 ? 512 : t);
}

// launch the policy evaluation with the mapping that suits the particle count
static int launch_policy(const McpPolicy& pol, const McpModel& mdl, const McpNoise& nz, int M, int Mg, int t, int tm,
                         const double* pol_in_t, const double* x_t, double* u_t, double* Xs, cudaStream_t st) {
  if (Mg <= 2048)  // chosen from the GLOBAL particle count: shards of one rollout must add the basis functions in the same order
    policy_fwd_block_kernel<<<M, policy_block_threads(pol.nb), 0, st>>>(pol, mdl, nz, M, t, tm, pol_in_t, x_t, u_t, Xs);
  else
    policy_fwd_kernel<<<cdiv(M, 8), 256, 0, st>>>(pol, mdl, nz, M, t, tm, pol_in_t, x_t, u_t, Xs);
  MCP_LAUNCH_CHECK();
  return MCP_OK;
}

// delta = mean + sqrt(var) eps; integrate; checkpoint J = d(delta)/d(gp input); simulated measurement (4PMS).
// Model_learning.py:685-718 / :471-493; MC_PILCO.py:878-899.
__global__ void __launch_bounds__(128) integrate_kernel(const __grid_constant__ McpModel mdl, const __grid_constant__ McpMeas ms,
                                                        const __grid_constant__ McpNoise nz, int M, int t,
                                                        const double* __restrict__ x_t, const double* __restrict__ mean,
                                                        const double* __restrict__ var, const double* __restrict__ jmean,
                                                        const double* __restrict__ jvar, double* __restrict__ x_n,
                                                        double* __restrict__ jac_t, const double* __restrict__ polin_t,
                                                        double* __restrict__ polin_n, double* __restrict__ nv) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M) return;
  const int E = mdl.E, D = mdl.D, Ds = mdl.Ds;
  const double* x = x_t + (size_t)m * Ds;
  double* xn = x_n + (size_t)m * Ds;
  if (mdl.kind == 1)
    for (int j = 0; j < Ds; j++) xn[j] = 0.0;  // the reference starts from zeros (Model_learning.py:700)
  for (int e = 0; e < E; e++) {
    double mu = mean[(size_t)m * E + e], v = var[(size_t)m * E + e];
    double delta = mu, coef = 0.0;
    if (mdl.particle_pred) {
      double eps = nz.eps ? nz.eps[((size_t)t * M + m) * E + e] : rng_normal(noise_seed(nz), nz.particle_offset + (uint64_t)m, t, RNG_EPS, e);
      double sd = sqrt(v);
      delta = fma(sd, eps, mu);
      coef = eps / (2.0 * sd);
    }
    if (jac_t) {
      const double* jm = jmean + ((size_t)m * E + e) * D;
      const double* jv = jvar + ((size_t)m * E + e) * D;
      double* jo = jac_t + ((size_t)m * E + e) * D;
      for (int d = 0; d < D; d++) jo[d] = fma(coef, jv[d], jm[d]);
    }
    if (mdl.kind == 1) {
      int iv = mdl.vel_idx[e], ip = mdl.pos_idx[e];
      xn[iv] = x[iv] + delta;
      xn[ip] = x[ip] + mdl.T * x[iv] + 0.5 * mdl.T * delta;
    } else {
      xn[e] = x[e] + delta;
    }
  }
  if (ms.enabled) {
    // noisy positions, finite-difference velocity, first-order low-pass (MC_PILCO.py:881-899)
    const double* pp = polin_t + (size_t)m * Ds;
    double* pn = polin_n + (size_t)m * Ds;
    for (int j = 0; j < Ds; j++) pn[j] = xn[j];
    for (int i = 0; i < ms.n_pos; i++) {
      int ip = ms.pos_idx[i], iv = ms.vel_idx[i];
      double e = nz.meas_eps ? nz.meas_eps[((size_t)t * M + m) * ms.n_pos + i]
                             : rng_normal(noise_seed(nz), nz.particle_offset + (uint64_t)m, t, RNG_MEAS, i);
      double np_old = pp[ip], mv_old = pp[iv];
      double np_new = fma(ms.std_pos[i], e, xn[ip]);
      double nv_old = nv[(size_t)m * ms.n_pos + i];
      double nv_new = (np_new - np_old) / ms.T;
      double mv_new = (ms.b0 * nv_new + ms.b1 * nv_old - ms.a1 * mv_old) / ms.a0;
      nv[(size_t)m * ms.n_pos + i] = nv_new;
      pn[ip] = np_new;
      pn[iv] = mv_new;
    }
  }
}

// initial particles from Philox (MC_PILCO.py:635-657); stream RNG_X0, "time" index 0
__global__ void init_particles_kernel(int kind, const double* __restrict__ a, const double* __restrict__ b, int n_modes, int M, int Ds,
                                      uint64_t seed, uint64_t offset, const uint64_t* __restrict__ seed_dev, double* __restrict__ x0) {
  int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M) return;
  if (seed_dev) seed += __ldg(seed_dev);
  uint64_t pid = offset + (uint64_t)m;
  int k = 0;
  if (n_modes > 1) {
    Philox4 q = philox4x32_10(seed, (uint32_t)pid, (uint32_t)(pid >> 32), (uint32_t)RNG_X0 << 24, 0xFFFFFFFFu);
    k = (int)(((uint64_t)q.v[0] * (uint64_t)n_modes) >> 32);
  }
  for (int j = 0; j < Ds; j++) {
    double lo = a[(size_t)k * Ds + j], hi = b[(size_t)k * Ds + j];
    if (kind == 0) {
      x0[(size_t)m * Ds + j] = fma(hi, rng_normal(seed, pid, 0, RNG_X0, j), lo);
    } else {
      Philox4 q = philox4x32_10(seed, (uint32_t)pid, (uint32_t)(pid >> 32), (uint32_t)RNG_X0 << 24, (uint32_t)j);
      x0[(size_t)m * Ds + j] = fma(hi - lo, u01(q.v[0], q.v[1]), lo);
    }
  }
}

// The same step with one WARP per particle (lanes over outputs, then over the E x D checkpoint entries): used for small particle
// counts, where a thread per particle leaves the GPU idle behind a serial E x D loop.
__device__ __forceinline__ void integrate_warp_body(const McpModel& mdl, const McpMeas& ms, const McpNoise& nz, int M, int t, int m, int lane,
                                                    const double* __restrict__ x_t, const double* __restrict__ mean,
                                                    const double* __restrict__ var, const double* __restrict__ jmean,
                                                    const double* __restrict__ jvar, double* __restrict__ x_n,
                                                    double* __restrict__ jac_t, const double* __restrict__ polin_t,
                                                    double* __restrict__ polin_n, double* __restrict__ nv) {
  const int E = mdl.E, D = mdl.D, Ds = mdl.Ds;
  const double* x = x_t + (size_t)m * Ds;
  double* xn = x_n + (size_t)m * Ds;
  double delta = 0.0, coef = 0.0;
  if (lane < E) {
    const double mu = mean[(size_t)m * E + lane], v = var[(size_t)m * E + lane];
    delta = mu;
    if (mdl.particle_pred) {
      const double eps = nz.eps ? nz.eps[((size_t)t * M + m) * E + lane] : rng_normal(noise_seed(nz), nz.particle_offset + (uint64_t)m, t, RNG_EPS, lane);
      const double sd = sqrt(v);
      delta = fma(sd, eps, mu);
      coef = eps / (2.0 * sd);
    }
  }
  if (jac_t) {
    const size_t base = (size_t)m * E * D;
    const int n = E * D;
    for (int i0 = 0; i0 < n; i0 += 32) {
      const int idx = i0 + lane, e = min(idx, n - 1) / D;
      const double ce = __shfl_sync(0xffffffffu, coef, e);
      if (idx < n) jac_t[base + idx] = fma(ce, jvar[base + idx], jmean[base + idx]);
    }
  }
  if (mdl.kind == 1) {
    if (lane < Ds) xn[lane] = 0.0;  // the reference starts from zeros (Model_learning.py:700)
    __syncwarp();
    if (lane < E) {
      const int iv = mdl.vel_idx[lane], ip = mdl.pos_idx[lane];
      xn[iv] = x[iv] + delta;
      xn[ip] = x[ip] + mdl.T * x[iv] + 0.5 * mdl.T * delta;
    }
  } else if (lane < E) {
    xn[lane] = x[lane] + delta;
  }
  if (ms.enabled) {
    __syncwarp();
    const double* pp = polin_t + (size_t)m * Ds;
    double* pn = polin_n + (size_t)m * Ds;
    if (lane < Ds) pn[lane] = xn[lane];
    __syncwarp();
    if (lane < ms.n_pos) {
      const int i = lane, ip = ms.pos_idx[i], iv = ms.vel_idx[i];
      const double e = nz.meas_eps ? nz.meas_eps[((size_t)t * M + m) * ms.n_pos + i]
                                   : rng_normal(noise_seed(nz), nz.particle_offset + (uint64_t)m, t, RNG_MEAS, i);
      const double np_old = pp[ip], mv_old = pp[iv];
      const double np_new = fma(ms.std_pos[i], e, xn[ip]);
      const double nv_old = nv[(size_t)m * ms.n_pos + i];
      const double nv_new = (np_new - np_old) / ms.T;
      const double mv_new = (ms.b0 * nv_new + ms.b1 * nv_old - ms.a1 * mv_old) / ms.a0;
      nv[(size_t)m * ms.n_pos + i] = nv_new;
      pn[ip] = np_new;
      pn[iv] = mv_new;
    }
  }
}

__global__ void __launch_bounds__(256) integrate_warp_kernel(const __grid_constant__ McpModel mdl, const __grid_constant__ McpMeas ms,
                                                             const __grid_constant__ McpNoise nz, int M, int t,
                                                             const double* __restrict__ x_t, const double* __restrict__ mean,
                                                             const double* __restrict__ var, const double* __restrict__ jmean,
                                                             const double* __restrict__ jvar, double* __restrict__ x_n,
                                                             double* __restrict__ jac_t, const double* __restrict__ polin_t,
                                                             double* __restrict__ polin_n, double* __restrict__ nv) {
  const int m = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (m >= M) return;
  integrate_warp_body(mdl, ms, nz, M, t, m, lane, x_t, mean, var, jmean, jvar, x_n, jac_t, polin_t, polin_n, nv);
}

// Small particle counts: the model step t -> t+1 and the policy evaluation at t+1 of one particle in ONE block (warp 0 integrates, a
// block barrier, then all threads evaluate the policy): one launch boundary less on the per-step chain.
__global__ void __launch_bounds__(512) integrate_policy_block_kernel(const __grid_constant__ McpModel mdl, const __grid_constant__ McpMeas ms,
                                                                     const __grid_constant__ McpNoise nz, const __grid_constant__ McpPolicy pol,
                                                                     int M, int t, const double* __restrict__ x_t,
                                                                     const double* __restrict__ mean, const double* __restrict__ var,
                                                                     const double* __restrict__ jmean, const double* __restrict__ jvar,
                                                                     double* __restrict__ x_n, double* __restrict__ jac_t,
                                                                     const double* __restrict__ polin_t, double* __restrict__ polin_n,
                                                                     double* __restrict__ nv, double* __restrict__ u_n, double* __restrict__ Xs) {
  if (threadIdx.x < 32)
    integrate_warp_body(mdl, ms, nz, M, t, (int)blockIdx.x, (int)threadIdx.x, x_t, mean, var, jmean, jvar, x_n, jac_t, polin_t, polin_n, nv);
  __syncthreads();  // the block's own global writes (x_{t+1}, the policy input) are visible to it after the barrier
  policy_block_body(pol, mdl, nz, M, t + 1, t + 1, ms.enabled ? polin_n : x_n, x_n, u_n, Xs);
}

__global__ void init_nv_kernel(const __grid_constant__ McpMeas ms, int M, int Ds, const double* __restrict__ x0, double* __restrict__ nv) {
  int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M) return;
  for (int i = 0; i < ms.n_pos; i++) nv[(size_t)m * ms.n_pos + i] = x0[(size_t)m * Ds + ms.vel_idx[i]];
}

__global__ void __launch_bounds__(256) cost_kernel(const __grid_constant__ McpCost c, int M, int H, int Ds,
                                                   const double* __restrict__ states, double* __restrict__ costs) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)M * H) return;
  int t = (int)(i / M);
  costs[i] = cost_value(c, states + i * Ds, t, Ds);
}

// per time step: mean and M2 = sum (c - mean)^2 over particles (two passes, fixed summation order)
__global__ void __launch_bounds__(256) cost_stats_kernel(int M, const double* __restrict__ costs, double* __restrict__ stats) {
  __shared__ double red[8];
  __shared__ double s_mean;
  const int t = blockIdx.x, tid = threadIdx.x;
  const double* c = costs + (size_t)t * M;
  double a = 0.0;
  for (int m = tid; m < M; m += 256) a += c[m];
  a = warp_sum(a);
  if ((tid & 31) == 0) red[tid >> 5] = a;
  __syncthreads();
  if (tid == 0) {
    double s = 0.0;
    for (int i = 0; i < 8; i++) s += red[i];
    s_mean = s / M;
  }
  __syncthreads();
  double mean = s_mean, q = 0.0;
  for (int m = tid; m < M; m += 256) {
    double d = c[m] - mean;
    q = fma(d, d, q);
  }
  q = warp_sum(q);
  __syncthreads();
  if ((tid & 31) == 0) red[tid >> 5] = q;
  __syncthreads();
  if (tid == 0) {
    double s = 0.0;
    for (int i = 0; i < 8; i++) s += red[i];
    stats[2 * t] = mean;
    stats[2 * t + 1] = s;
  }
}

// Expected_cost.forward: sum_t mean_t and sum_t unbiased std_t.  Cost_function.py:33-36
__global__ void cost_final_kernel(int M, int H, const double* __restrict__ stats, double* __restrict__ out) {
  if (threadIdx.x != 0) return;
  double a = 0.0, b = 0.0;
  for (int t = 0; t < H; t++) {
    a += stats[2 * t];
    b += sqrt(stats[2 * t + 1] / (double)(M - 1));
  }
  out[0] = a;
  out[1] = b;
}

// ------------------------------------------------------------------------------------------------
// backward: reverse sweep over the horizon, one CTA per particle (grid-strided).
// The adjoint recursion lambda_{t+1} -> lambda_t is one serial chain per particle, so the kernel is organised around the length of
// that chain and nothing else:
//   * the first ceil(nb / 32) warps own one policy basis function per thread; one extra warp (the "chain warp") carries the adjoints,
//     lane j holding component j;
//   * everything that does not depend on the incoming adjoint is computed AHEAD of the chain by the basis threads while the chain
//     warp works: the checkpoint of step t-5 streams global -> shared (cp.async, ring of 8 slots), the policy features, the cost
//     gradient and the sines / cosines of step t-2 are derived from the ring (ring of 4), and the basis activations h_b (exp, dropout
//     draw) of step t-1 sit in a register when the chain reaches that step;
//   * per step two block barriers remain: [basis part of the policy adjoint] Z [chain warp: cross-warp sums, policy-input adjoint,
//     measurement model, model step t-1 -> adjoint of u_{t-1}] Y.
// Reference: the autograd graph of apply_policy (policy_learning/MC_PILCO.py:615-674, :808-906) walked by cost.backward() (:522).
// ------------------------------------------------------------------------------------------------
constexpr int BW_RING = 8, BW_AUX = 4, BW_LAG = 5;

// Sums N = 8 / 16 / 32 per-lane values over the warp with N - 1 + (5 - log2 N) shuffles instead of 5 N: each butterfly level halves the
// number of values a lane still carries.  Afterwards v[0] of lane l holds the warp total of value l >> (5 - log2 N) (the lanes that share
// those upper bits all hold it).  Fixed order, so the result is reproducible.
template <int N>
__device__ __forceinline__ void warp_sum_multi(double (&v)[N], int lane) {
  static_assert(N == 8 || N == 16 || N == 32, "warp_sum_multi: 8, 16 or 32 values");
  int offset = 16;
#pragma unroll
  for (int n = N; n > 1; n >>= 1, offset >>= 1) {
    const bool hi = (lane & offset) != 0;
#pragma unroll
    for (int j = 0; j < n / 2; j++) {
      const double send = hi ? v[j] : v[j + n / 2], keep = hi ? v[j + n / 2] : v[j];
      v[j] = keep + __shfl_xor_sync(0xffffffffu, send, offset);
    }
  }
#pragma unroll
  for (; offset >= 1; offset >>= 1) v[0] += __shfl_xor_sync(0xffffffffu, v[0], offset);
}

template <int DPT, int DUT, int NT, int NCTA>
__global__ void __launch_bounds__(NT, NCTA) rollout_bwd_kernel(const __grid_constant__ McpRollout r, const __grid_constant__ McpRolloutGrad g,
                                                           double* __restrict__ partials, double* __restrict__ g_x0) {
  extern __shared__ double bw_ring[];  // [BW_RING][x | policy input | grad_states | u | grad_inputs | Jacobian rows]
  const McpModel& mdl = r.model;
  const McpPolicy& pol = r.policy;
  const McpMeas& ms = r.meas;
  const int M = r.M, H = r.H, Ds = mdl.Ds, Du = mdl.Du, E = mdl.E, D = mdl.D, nb = pol.nb, Dp = pol.Dp;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nbw = (nb + 31) >> 5, nbt = nbw * 32;  // basis warps / threads; warp nbw is the chain warp
  const bool chain = warp == nbw;
  const int b = tid;
  const bool has_b = b < nb;
  const int o_px = Ds, o_gs = 2 * Ds, o_u = 3 * Ds, o_gi = 3 * Ds + Du, o_J = 3 * Ds + 2 * Du, slot_n = o_J + E * D;

  __shared__ double s_il[MCP_MAX_DP];
  __shared__ double s_z[BW_AUX][MCP_MAX_DP], s_lam0[BW_AUX][MCP_MAX_DS];
  __shared__ double s_msin[BW_AUX][MCP_MAX_DS], s_mcos[BW_AUX][MCP_MAX_DS], s_psin[BW_AUX][MCP_MAX_DS], s_pcos[BW_AUX][MCP_MAX_DS];
  __shared__ double s_la[MCP_MAX_DU];
  __shared__ double s_red[16][MCP_MAX_DP];
  __shared__ int s_active;

  if (tid < Dp) s_il[tid] = exp(-pol.log_ls[tid]);
  // centres of this thread's basis function: registers, or — widest instance (up to 32 features: centres + their gradient accumulators
  // + the per-step terms would be 96 doubles per thread and spilled) — a [feature][thread] array in shared memory behind the ring
  constexpr bool CB_SMEM = DPT > 16;
  constexpr int CBR = CB_SMEM ? 1 : DPT;
  double cb_reg[CBR], gc[DPT], wb[DUT], gw[DUT];
  double* const s_cb = bw_ring + (size_t)BW_RING * slot_n;  // [Dp][blockDim.x] (CB_SMEM only)
#define MCP_CBV(j) (CB_SMEM ? s_cb[(size_t)(j) * nthr + tid] : cb_reg[CB_SMEM ? 0 : (j)])
  const int nthr = blockDim.x;
#pragma unroll
  for (int j = 0; j < DPT; j++) {
    const double c = (has_b && j < Dp) ? pol.centers[(size_t)b * Dp + j] : 0.0;
    if (CB_SMEM) { if (j < Dp) s_cb[(size_t)j * nthr + tid] = c; }
    else cb_reg[CB_SMEM ? 0 : j] = c;
    gc[j] = 0.0;
  }
#pragma unroll
  for (int k = 0; k < DUT; k++) { wb[k] = (has_b && k < Du) ? pol.W[(size_t)k * nb + b] : 0.0; gw[k] = 0.0; }
  const bool drop = dropout_active(pol, r.noise);
  const double keep_scale = drop ? 1.0 / (1.0 - r.noise.p_dropout) : 1.0;
  const double cost_w = (r.cost.kind != 0) ? g.grad_cost / (double)M : 0.0;  // adds to grad_states / grad_inputs when both are given
  const double* polin = (ms.enabled && r.pol_in) ? r.pol_in : r.states;
  // chain-warp registers: lane j carries component j
  double glz = 0.0, gbias = 0.0;  // log-lengthscale gradient (first half, see below), bias gradient
  // where component `lane` of the state sits in the index lists of the model and the policy (-1: nowhere; the lists hold each state
  // component at most once), looked up once so that the per-step chain has no loops over them
  int c_vel = -1, c_pos = -1, c_partner = 0, c_mna = -1, c_ma = -1, c_pna = -1, c_pa = -1, e_iv = 0, e_ip = 0;
  double c_isc0 = 0.0, c_isc1 = 0.0, c_isc2 = 0.0, c_umax = 1.0;
  if (chain) {
    if (mdl.kind == 1) {
      for (int e = 0; e < E; e++) {
        if (mdl.vel_idx[e] == lane) { c_vel = e; c_partner = mdl.pos_idx[e]; }
        if (mdl.pos_idx[e] == lane) c_pos = e;
      }
      if (lane < E) { e_iv = mdl.vel_idx[lane]; e_ip = mdl.pos_idx[lane]; }
    }
    if (mdl.use_trig) {
      for (int i = 0; i < mdl.n_na; i++) if (mdl.na_idx[i] == lane) c_mna = i;
      for (int i = 0; i < mdl.n_a; i++) if (mdl.a_idx[i] == lane) c_ma = i;
    }
    if (pol.kind == 1) {
      for (int i = 0; i < pol.n_na; i++) if (pol.na_idx[i] == lane) { c_pna = i; c_isc0 = pol.inv_scale[i]; }
      for (int i = 0; i < pol.n_a; i++)
        if (pol.a_idx[i] == lane) { c_pa = i; c_isc1 = pol.inv_scale[pol.n_na + i]; c_isc2 = pol.inv_scale[pol.n_na + pol.n_a + i]; }
    } else if (lane < Ds) {
      c_isc0 = pol.inv_scale[lane];
      if (pol.kind == 2) c_isc1 = pol.inv_scale[Ds + lane];
    }
    if (lane < Du && pol.squash) c_umax = pol.u_max[lane];
  }
  __syncthreads();

  for (int m = blockIdx.x; m < M; m += gridDim.x) {
    // ---- helpers --------------------------------------------------------------------------------------------------------------
    // checkpoint of step tt: global -> ring slot, asynchronously (basis threads; one commit group per call, empty past the start)
    auto issue = [&](int tt) {
      if (tt >= 0) {
        double* slot = bw_ring + (size_t)(tt & (BW_RING - 1)) * slot_n;
        const size_t row = (size_t)tt * M + m;
        for (int i = (tid >= nbt - 32) ? tid - (nbt - 32) : tid + 32; i < slot_n; i += nbt) {  // the last basis warp first: warp 0 has the heaviest role above
          const double* src = nullptr;
          if (i < o_px) src = r.states + row * Ds + i;
          else if (i < o_gs) src = polin + row * Ds + (i - o_px);
          else if (i < o_u) src = g.grad_states ? g.grad_states + row * Ds + (i - o_gs) : nullptr;
          else if (i < o_gi) src = r.inputs + row * Du + (i - o_u);
          else if (i < o_J) src = g.grad_inputs ? g.grad_inputs + row * Du + (i - o_gi) : nullptr;
          else src = (tt < H - 1) ? r.jac + row * E * D + (i - o_J) : nullptr;
          cp_async8(slot + i, src ? src : r.states, src ? 8 : 0);
        }
      }
      cp_async_commit();
    };
    // adjoint-independent quantities of step tt from its ring slot (basis threads, one role each)
    auto aux = [&](int tt) {
      if (tt < 0) return;
      const double* slot = bw_ring + (size_t)(tt & (BW_RING - 1)) * slot_n;
      const int a = tt & (BW_AUX - 1);
      const int n_ma = mdl.use_trig ? mdl.n_a : 0, n_pa = (pol.kind == 1) ? pol.n_a : 0;
      const int nroles = Dp + 1 + n_ma + n_pa;
      // role r -> lane r / nbw of warp r % nbw: the divergent roles (cos / sin / cost gradient) run in different warps, in parallel
      for (int role = lane * nbw + warp; role < nroles; role += nbt) {
        if (role < Dp) {
          s_z[a][role] = policy_feature(pol, slot + o_px, tt, role);
        } else if (role == Dp) {  // adjoint of x_tt from the caller's gradient and the fused cost
          for (int j = 0; j < Ds; j++) s_lam0[a][j] = slot[o_gs + j];
          if (cost_w != 0.0) cost_grad_add(r.cost, slot, tt, Ds, cost_w, s_lam0[a]);
        } else if (role < Dp + 1 + n_ma) {
          const int i = role - Dp - 1;
          double sn, cs;
          sincos(slot[mdl.a_idx[i]], &sn, &cs);
          s_msin[a][i] = sn;
          s_mcos[a][i] = cs;
        } else {
          const int i = role - Dp - 1 - n_ma;
          double sn, cs;
          sincos(slot[o_px + pol.a_idx[i]], &sn, &cs);
          s_psin[a][i] = sn;
          s_pcos[a][i] = cs;
        }
      }
    };
    // activation of this thread's basis function at step tt (needs aux(tt))
    auto activation = [&](int tt) {
      double h = 0.0;
      if (has_b && tt >= 0) {
        const double* z = s_z[tt & (BW_AUX - 1)];
        double d = 0.0;
#pragma unroll
        for (int j = 0; j < DPT; j++)
          if (j < Dp) { double q = (z[j] - MCP_CBV(j)) * s_il[j]; d = fma(q, q, d); }
        h = exp(-d);
        if (drop) h = keep_unit(r.noise, M, nb, tt, tt, m, b) ? h * keep_scale : 0.0;
      }
      return h;
    };
    // chain warp, stage A of step tt: adjoint of x_tt from the cost and from the model step tt -> tt+1 (lane j: component j, returned);
    // adjoint of u_tt -> s_la, s_active
    // (everything the lanes exchange goes through shuffles: ln is the adjoint x_{tt+1} received, component `lane`)
    auto chain_A = [&](int tt, double ln) {
      const double* slot = bw_ring + (size_t)(tt & (BW_RING - 1)) * slot_n;
      const int a = tt & (BW_AUX - 1);
      double lam = lane < Ds ? s_lam0[a][lane] : 0.0;
      double lu = lane < Du ? slot[o_gi + lane] : 0.0;
      if (tt < H - 1) {
        // adjoint of the GP output e in lane e; lx[d] = sum_e ld_e J[e][d] in lane d
        double ld = ln;
        if (mdl.kind == 1) {
          const double a_v = __shfl_sync(0xffffffffu, ln, e_iv), a_p = __shfl_sync(0xffffffffu, ln, e_ip);
          ld = a_v + 0.5 * mdl.T * a_p;
          const double part = __shfl_sync(0xffffffffu, ln, c_partner);
          if (c_vel >= 0) lam += ln + mdl.T * part;
          if (c_pos >= 0) lam += ln;
        } else if (lane < E) {
          lam += ln;
        }
        double lx = 0.0;
        const double* Jd = slot + o_J + (lane < D ? lane : 0);
        for (int e = 0; e < E; e++) lx = fma(__shfl_sync(0xffffffffu, ld, e), Jd[e * D], lx);
        if (mdl.use_trig) {
          const int n_na = mdl.n_na, n_a = mdl.n_a;
          const double x_na = __shfl_sync(0xffffffffu, lx, c_mna >= 0 ? c_mna : 0);
          const double x_c = __shfl_sync(0xffffffffu, lx, (n_na + (c_ma >= 0 ? c_ma : 0)) & 31);
          const double x_s = __shfl_sync(0xffffffffu, lx, (n_na + n_a + (c_ma >= 0 ? c_ma : 0)) & 31);
          const double x_u = __shfl_sync(0xffffffffu, lx, (n_na + 2 * n_a + lane) & 31);
          if (c_mna >= 0) lam += x_na;
          if (c_ma >= 0) lam += x_c * s_mcos[a][c_ma] - x_s * s_msin[a][c_ma];
          if (lane < Du) lu += x_u;
        } else {
          const double x_u = __shfl_sync(0xffffffffu, lx, (Ds + lane) & 31);
          if (lane < Ds) lam += lx;
          if (lane < Du) lu += x_u;
        }
      }
      double la = 0.0;
      if (lane < Du) {
        la = lu;
        if (pol.squash) { double q = slot[o_u + lane] / c_umax; la *= (1.0 - q * q); }
        s_la[lane] = la;
        gbias += la;
      }
      const unsigned act = __ballot_sync(0xffffffffu, la != 0.0);
      if (lane == 0) s_active = act != 0u;
      return lam;
    };

    // ---- pipeline fill ----------------------------------------------------------------------------------------------------------
    double lam = 0.0, h = 0.0;   // chain: adjoint of x_t after stage A; basis: activation at the chain's current step
    double lnv = 0.0, lmv = 0.0, lnp = 0.0;  // 4PMS carried adjoints of position pair i, replicated... (lane i of the chain warp)
    if (!chain) {
#pragma unroll
      for (int k = 0; k < BW_LAG; k++) issue(H - 1 - k);
      cp_async_wait<BW_LAG - 2>();  // steps H-1 and H-2 have landed
    }
    __syncthreads();
    if (!chain) { aux(H - 1); aux(H - 2); }
    __syncthreads();
    if (chain) {
      lam = chain_A(H - 1, 0.0);
    } else {
      h = activation(H - 1);
      cp_async_wait<2>();  // step H-3
    }
    __syncthreads();

    for (int t = H - 1; t >= 0; t--) {
      const double* z = s_z[t & (BW_AUX - 1)];
      const bool active = s_active != 0;
      // ---- basis threads: policy adjoint of step t, thread b owns basis function b ----
      if (!chain && active) {
        double lh = 0.0;
#pragma unroll
        for (int k = 0; k < DUT; k++)
          if (k < Du) { gw[k] = fma(s_la[k], h, gw[k]); lh = fma(s_la[k], wb[k], lh); }
        const double ld_b = -h * lh;
        constexpr int CH = DPT > 16 ? 16 : DPT;  // features per butterfly (the widest instance takes two, to stay in registers)
        constexpr int SH = CH == 8 ? 2 : 1;
#pragma unroll
        for (int j0 = 0; j0 < DPT; j0 += CH) {
          double cz[CH];
#pragma unroll
          for (int jj = 0; jj < CH; jj++) {
            const int j = j0 + jj;
            cz[jj] = (j < Dp) ? ld_b * 2.0 * (z[j] - MCP_CBV(j)) * s_il[j] * s_il[j] : 0.0;  // d/dz_j ; d/dc_bj = -cz
            gc[j] -= cz[jj];
          }
          warp_sum_multi<CH>(cz, lane);
          if ((lane & ((1 << SH) - 1)) == 0 && j0 + (lane >> SH) < Dp) s_red[warp][j0 + (lane >> SH)] = cz[0];
        }
      }
      __syncthreads();  // Z
      if (chain) {
        // ---- adjoint of the policy input -> adjoint of x_t (through the measurement model if any) ----
        double lz = 0.0;
        if (active && lane < Dp) {
          for (int w2 = 0; w2 < nbw; w2++) lz += s_red[w2][lane];
          glz -= z[lane] * lz;  // log-lengthscale gradient, first half (see below)
        }
        double lp = 0.0;
        {
          const int a = t & (BW_AUX - 1);
          if (pol.kind == 1) {
            const int n_na = pol.n_na, n_a = pol.n_a;
            const double z_na = __shfl_sync(0xffffffffu, lz, c_pna >= 0 ? c_pna : 0);
            const double z_c = __shfl_sync(0xffffffffu, lz, (n_na + (c_pa >= 0 ? c_pa : 0)) & 31);
            const double z_s = __shfl_sync(0xffffffffu, lz, (n_na + n_a + (c_pa >= 0 ? c_pa : 0)) & 31);
            if (c_pna >= 0) lp += z_na * c_isc0;
            if (c_pa >= 0) lp += -z_c * c_isc1 * s_psin[a][c_pa] + z_s * c_isc2 * s_pcos[a][c_pa];
          } else if (pol.kind == 2) {
            const double z_t = __shfl_sync(0xffffffffu, lz, (Ds + lane) & 31);
            if (lane < Ds) lp += lz * c_isc0 - z_t * c_isc1;
          } else {
            if (lane < Ds) lp += lz * c_isc0;
          }
        }
        if (ms.enabled) {
          for (int i = 0; i < ms.n_pos; i++) {   // lane i carries the filter adjoints of pair i
            const int ip = ms.pos_idx[i], iv = ms.vel_idx[i];
            const double c_lnv = __shfl_sync(0xffffffffu, lnv, i), c_lmv = __shfl_sync(0xffffffffu, lmv, i), c_lnp = __shfl_sync(0xffffffffu, lnp, i);
            double a_lnp = c_lnp + __shfl_sync(0xffffffffu, lp, ip), a_lmv = c_lmv + __shfl_sync(0xffffffffu, lp, iv), a_lnv = c_lnv;
            if (lane == ip || lane == iv) lp = 0.0;
            if (t > 0) {
              a_lnv += ms.b0 / ms.a0 * a_lmv;
              const double n_lnv = ms.b1 / ms.a0 * a_lmv;   // carried to nv_{t-1}
              const double n_lmv = -ms.a1 / ms.a0 * a_lmv;  // carried to mv_{t-1}
              a_lnp += a_lnv / ms.T;
              const double n_lnp = -a_lnv / ms.T;           // carried to np_{t-1}
              if (lane == i) { lnv = n_lnv; lmv = n_lmv; lnp = n_lnp; }
              if (lane == ip) lam += a_lnp;
            } else {
              if (lane == ip) lam += a_lnp;
              if (lane == iv) lam += a_lnv + a_lmv;
            }
          }
        }
        lam += lp;   // = adjoint of x_t, complete
        if (t > 0) lam = chain_A(t - 1, lam);
      } else {
        // ---- ahead of the chain: activation of step t-1, derived quantities of step t-2, checkpoint of step t-5 ----
        h = activation(t - 1);
        aux(t - 2);
        issue(t - BW_LAG);
        cp_async_wait<2>();  // the checkpoint aux() reads one iteration from now has landed
      }
      __syncthreads();  // Y
    }
    if (chain && g_x0 != nullptr && lane < Ds) g_x0[(size_t)m * Ds + lane] = lam;
  }

  // ---- per-CTA partial gradients: [g_log_ls (Dp) | g_centers (nb*Dp) | g_W (Du*nb) | g_bias (Du)] ----
  // d/dlog l_j of ((z_j-c_bj)/l_j)^2 = -2 ((z_j-c_bj)/l_j)^2, hence
  //   g_logls_j = sum_steps sum_b [d/dc_bj contribution] (z_j - c_bj) = -sum_steps z_j lz_j - sum_b c_bj g_c[b][j]
  double* P = partials + (size_t)blockIdx.x * (Dp + (size_t)nb * Dp + (size_t)Du * nb + Du);
  if (!chain) {
    constexpr int CH = DPT > 16 ? 16 : DPT;
    constexpr int SH = CH == 8 ? 2 : 1;
#pragma unroll
    for (int j0 = 0; j0 < DPT; j0 += CH) {
      double cg[CH];
#pragma unroll
      for (int jj = 0; jj < CH; jj++) cg[jj] = (j0 + jj < Dp) ? MCP_CBV(j0 + jj) * gc[j0 + jj] : 0.0;
      warp_sum_multi<CH>(cg, lane);
      if ((lane & ((1 << SH) - 1)) == 0 && j0 + (lane >> SH) < Dp) s_red[warp][j0 + (lane >> SH)] = cg[0];
    }
  }
  __syncthreads();
  if (chain) {
    if (lane < Dp) {
      double v = 0.0;
      for (int w2 = 0; w2 < nbw; w2++) v += s_red[w2][lane];
      P[lane] = glz - v;
    }
    if (lane < Du) P[Dp + (size_t)nb * Dp + (size_t)Du * nb + lane] = gbias;
  }
  if (has_b) {
#pragma unroll
    for (int j = 0; j < DPT; j++)
      if (j < Dp) P[Dp + (size_t)b * Dp + j] = gc[j];
#pragma unroll
    for (int k = 0; k < DUT; k++)
      if (k < Du) P[Dp + (size_t)nb * Dp + (size_t)k * nb + b] = gw[k];
  }
}

#undef MCP_CBV

// out[i] = sum over CTAs of partials[cta][i] (fixed order -> bit-stable)
__global__ void reduce_partials_kernel(const double* __restrict__ partials, int ncta, int n, double* __restrict__ out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double a = 0.0;
  for (int c = 0; c < ncta; c++) a += partials[(size_t)c * n + i];
  out[i] = a;
}

__global__ void scatter_grads_kernel(const double* __restrict__ flat, int Dp, int nb, int Du, double* g_log_ls, double* g_centers,
                                     double* g_W, double* g_bias) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  int n = Dp + nb * Dp + Du * nb + Du;
  if (i >= n) return;
  double v = flat[i];
  if (i < Dp) { if (g_log_ls) g_log_ls[i] = v; return; }
  i -= Dp;
  if (i < nb * Dp) { if (g_centers) g_centers[i] = v; return; }
  i -= nb * Dp;
  if (i < Du * nb) { if (g_W) g_W[i] = v; return; }
  i -= Du * nb;
  if (g_bias) g_bias[i] = v;
}

// ------------------------------------------------------------------------------------------------
// stand-alone policy backward: the vector-Jacobian product of mcpilco_policy_forward (Policy.py:242-265,323-335,389-403 under
// autograd).  Threads own basis functions, as in policy_block_body; a CTA walks its particles one after the other, so that every
// thread keeps g_centers[b, :] and g_W[:, b] in registers and the particle sums need no atomics.  Per particle:
//   h_b (recomputed, same dropout draw as the forward) -> [squash only: u = u_max tanh((W h + bias) / u_max)] ->
//   la = g_u (1 - (u / u_max)^2) -> g_W += la h^T, dL/dd_b = -h_b <la, W[:, b]> -> d/dz by a butterfly per warp -> warp 0: dL/dx.
// The log-lengthscale gradient uses the identity of rollout_bwd_kernel: g_logls_j = -sum z_j lz_j - sum_b c_bj g_c[b][j].
// ------------------------------------------------------------------------------------------------
template <int DPT, int DUT>
__global__ void __launch_bounds__(512) policy_bwd_kernel(const __grid_constant__ McpPolicy pol, const __grid_constant__ McpNoise nz, int M, int t,
                                                         const double* __restrict__ x, const double* __restrict__ g_u,
                                                         double* __restrict__ g_x, double* __restrict__ partials) {
  extern __shared__ double s_cb[];  // [Dp][blockDim.x] centres, then [Du][blockDim.x] weights of each thread's basis function
  __shared__ double s_il[MCP_MAX_DP], s_z[MCP_MAX_DP];
  __shared__ double s_part[16][MCP_MAX_DU], s_la[MCP_MAX_DU];
  __shared__ double s_red[16][MCP_MAX_DP];
  const int nb = pol.nb, Dp = pol.Dp, Du = pol.Du, Ds = pol.Ds;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5, nthr = blockDim.x;
  const int b = tid;
  const bool has_b = b < nb;
  if (tid < Dp) s_il[tid] = exp(-pol.log_ls[tid]);
  double* const s_wb = s_cb + (size_t)Dp * nthr;
  double gc[DPT], gw[DUT];
#pragma unroll
  for (int j = 0; j < DPT; j++) {
    if (j < Dp) s_cb[(size_t)j * nthr + tid] = has_b ? pol.centers[(size_t)b * Dp + j] : 0.0;
    gc[j] = 0.0;
  }
#pragma unroll
  for (int k = 0; k < DUT; k++) {
    if (k < Du) s_wb[(size_t)k * nthr + tid] = has_b ? pol.W[(size_t)k * nb + b] : 0.0;
    gw[k] = 0.0;
  }
  const bool drop = dropout_active(pol, nz);
  const double keep_scale = drop ? 1.0 / (1.0 - nz.p_dropout) : 1.0;
  // warp 0: lane j carries the log-lengthscale gradient j (first half), lane k the bias gradient k; and where state component `lane`
  // sits in the feature lists (-1: nowhere)
  double glz = 0.0, gbias = 0.0;
  int c_pna = -1, c_pa = -1;
  if (warp == 0 && pol.kind == 1) {
    for (int i = 0; i < pol.n_na; i++) if (pol.na_idx[i] == lane) c_pna = i;
    for (int i = 0; i < pol.n_a; i++) if (pol.a_idx[i] == lane) c_pa = i;
  }
  __syncthreads();

  for (int m = blockIdx.x; m < M; m += gridDim.x) {
    const double* xm = x + (size_t)m * Ds;
    if (tid < Dp) s_z[tid] = policy_feature(pol, xm, t, tid);
    __syncthreads();
    double h = 0.0;
    if (has_b) {
      double d = 0.0;
#pragma unroll 4
      for (int j = 0; j < Dp; j++) { const double q = (s_z[j] - s_cb[(size_t)j * nthr + tid]) * s_il[j]; d = fma(q, q, d); }
      h = exp(-d);
      if (drop) h = keep_unit(nz, M, nb, 0, t, m, b) ? h * keep_scale : 0.0;
    }
    if (pol.squash) {  // the squash derivative needs the forward output
#pragma unroll
      for (int k = 0; k < DUT; k++)
        if (k < Du) {
          const double v = warp_sum(s_wb[(size_t)k * nthr + tid] * h);
          if (lane == 0) s_part[warp][k] = v;
        }
    }
    __syncthreads();
    if (tid < Du) {
      double la = g_u[(size_t)m * Du + tid];
      if (pol.squash) {
        double v = 0.0;
        for (int i = 0; i < nw; i++) v += s_part[i][tid];  // fixed order
        if (pol.has_bias) v += pol.bias[tid];
        const double q = tanh(v / pol.u_max[tid]);
        la *= 1.0 - q * q;
      }
      s_la[tid] = la;
      gbias += la;
    }
    __syncthreads();
    double lh = 0.0;
#pragma unroll
    for (int k = 0; k < DUT; k++)
      if (k < Du) { gw[k] = fma(s_la[k], h, gw[k]); lh = fma(s_la[k], s_wb[(size_t)k * nthr + tid], lh); }
    const double ld_b = -h * lh;  // dL/dd_b
#pragma unroll
    for (int j0 = 0; j0 < DPT; j0 += 8) {
      double cz[8];
#pragma unroll
      for (int jj = 0; jj < 8; jj++) {
        const int j = j0 + jj;
        cz[jj] = (j < Dp) ? ld_b * 2.0 * (s_z[j] - s_cb[(size_t)j * nthr + tid]) * s_il[j] * s_il[j] : 0.0;  // d/dz_j ; d/dc_bj = -cz
        gc[j] -= cz[jj];
      }
      warp_sum_multi<8>(cz, lane);
      if ((lane & 3) == 0 && j0 + (lane >> 2) < Dp) s_red[warp][j0 + (lane >> 2)] = cz[0];
    }
    __syncthreads();
    if (warp == 0) {
      double lz = 0.0;  // dL/dz_lane
      if (lane < Dp) {
        for (int w2 = 0; w2 < nw; w2++) lz += s_red[w2][lane];
        glz -= s_z[lane] * lz;
      }
      if (g_x != nullptr) {
        double gx = 0.0;
        if (pol.kind == 1) {
          const int n_na = pol.n_na, n_a = pol.n_a;
          const double z_na = __shfl_sync(0xffffffffu, lz, c_pna >= 0 ? c_pna : 0);
          const double z_c = __shfl_sync(0xffffffffu, lz, (n_na + (c_pa >= 0 ? c_pa : 0)) & 31);
          const double z_s = __shfl_sync(0xffffffffu, lz, (n_na + n_a + (c_pa >= 0 ? c_pa : 0)) & 31);
          if (c_pna >= 0) gx += z_na * pol.inv_scale[c_pna];
          if (c_pa >= 0) {
            double sn, cs;
            sincos(xm[lane], &sn, &cs);
            gx += -z_c * pol.inv_scale[n_na + c_pa] * sn + z_s * pol.inv_scale[n_na + n_a + c_pa] * cs;
          }
        } else if (pol.kind == 2) {
          const double z_t = __shfl_sync(0xffffffffu, lz, (Ds + lane) & 31);
          if (lane < Ds) gx = lz * pol.inv_scale[lane] - z_t * pol.inv_scale[Ds + lane];
        } else if (lane < Ds) {
          gx = lz * pol.inv_scale[lane];
        }
        if (lane < Ds) g_x[(size_t)m * Ds + lane] = gx;
      }
      __syncwarp();
    }
  }

  // per-CTA partials in the layout of reduce_partials_kernel / scatter_grads_kernel: [g_log_ls | g_centers | g_W | g_bias]
  double* P = partials + (size_t)blockIdx.x * (Dp + (size_t)nb * Dp + (size_t)Du * nb + Du);
  __syncthreads();
#pragma unroll
  for (int j0 = 0; j0 < DPT; j0 += 8) {
    double cg[8];
#pragma unroll
    for (int jj = 0; jj < 8; jj++) cg[jj] = (j0 + jj < Dp) ? s_cb[(size_t)(j0 + jj) * nthr + tid] * gc[j0 + jj] : 0.0;
    warp_sum_multi<8>(cg, lane);
    if ((lane & 3) == 0 && j0 + (lane >> 2) < Dp) s_red[warp][j0 + (lane >> 2)] = cg[0];
  }
  __syncthreads();
  if (warp == 0) {
    if (lane < Dp) {
      double v = 0.0;
      for (int w2 = 0; w2 < nw; w2++) v += s_red[w2][lane];
      P[lane] = glz - v;
    }
    if (lane < Du) P[Dp + (size_t)nb * Dp + (size_t)Du * nb + lane] = gbias;
  }
  if (has_b) {
#pragma unroll
    for (int j = 0; j < DPT; j++)
      if (j < Dp) P[Dp + (size_t)b * Dp + j] = gc[j];
#pragma unroll
    for (int k = 0; k < DUT; k++)
      if (k < Du) P[Dp + (size_t)nb * Dp + (size_t)k * nb + b] = gw[k];
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
struct Workspace {
  double *Xs, *mean, *var, *jmean, *jvar, *nv, *stats, *partials, *flat, *scratch;
  size_t scratch_doubles;
  int bwd_ctas;
};

// side streams / events for running the per-output chains of a small rollout concurrently (one set per device)
struct Fan {
  cudaStream_t side[MCP_MAX_E];
  cudaEvent_t fork, join[MCP_MAX_E];
};
static Fan* get_fan(cudaStream_t st) {
  // one set per (device, launching stream): two host threads driving different streams never share the fork / join events
  static std::map<std::pair<int, cudaStream_t>, Fan*> fans;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
  std::lock_guard<std::mutex> lock(init_mutex());
  auto key = std::make_pair(dev, st);
  auto it = fans.find(key);
  if (it != fans.end()) return it->second;
  if (fans.size() >= 256) return nullptr;  // callers fall back to running the chains one after the other
  Fan* f = new Fan();
  bool ok = cudaEventCreateWithFlags(&f->fork, cudaEventDisableTiming) == cudaSuccess;
  for (int e = 1; e < MCP_MAX_E && ok; e++)
    ok = cudaStreamCreateWithFlags(&f->side[e], cudaStreamNonBlocking) == cudaSuccess &&
         cudaEventCreateWithFlags(&f->join[e], cudaEventDisableTiming) == cudaSuccess;
  if (!ok) return nullptr;
  fans[key] = f;
  return f;
}

static int bwd_grid(int M) {
  int sms = 148;
  int dev = 0;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  int g = sms * 4;  // 4 resident CTAs per SM hide the latency of the per-step dependency chain
  return M < g ? M : g;
}

static size_t fixed_doubles(int M, int H, int E, int D, int nb, int Dp, int Du, int npos, int ctas) {
  size_t nparam = (size_t)Dp + (size_t)nb * Dp + (size_t)Du * nb + Du;
  size_t n = 0;
  n += align_up((size_t)M * D, 32);          // Xs
  n += 2 * align_up((size_t)M * E, 32);      // mean, var
  n += 2 * align_up((size_t)M * E * D, 32);  // jmean, jvar
  n += align_up((size_t)M * (npos > 0 ? npos : 1), 32);
  n += align_up((size_t)2 * H, 32);
  n += align_up((size_t)ctas * nparam, 32);
  n += align_up(nparam, 32);
  return n;
}

static int carve(const McpRollout* r, Workspace& w) {
  const int M = r->M, H = r->H, E = r->model.E, D = r->model.D;
  const int nb = r->policy.nb, Dp = r->policy.Dp, Du = r->policy.Du, npos = r->meas.enabled ? r->meas.n_pos : 0;
  MCP_CHECK_ARG(r->workspace != nullptr, "rollout: workspace missing");
  w.bwd_ctas = bwd_grid(M);
  double* p = (double*)align_up((size_t)r->workspace, 256);
  size_t avail = (r->workspace_bytes - ((char*)p - (char*)r->workspace)) / sizeof(double);
  size_t need = fixed_doubles(M, H, E, D, nb, Dp, Du, npos, w.bwd_ctas);
  MCP_CHECK_ARG(avail > need + 1024, "rollout: workspace too small (%zu doubles, need > %zu)", avail, need + 1024);
  size_t nparam = (size_t)Dp + (size_t)nb * Dp + (size_t)Du * nb + Du;
  w.Xs = p; p += align_up((size_t)M * D, 32);
  w.mean = p; p += align_up((size_t)M * E, 32);
  w.var = p; p += align_up((size_t)M * E, 32);
  w.jmean = p; p += align_up((size_t)M * E * D, 32);
  w.jvar = p; p += align_up((size_t)M * E * D, 32);
  w.nv = p; p += align_up((size_t)M * (npos > 0 ? npos : 1), 32);
  w.stats = p; p += align_up((size_t)2 * H, 32);
  w.partials = p; p += align_up((size_t)w.bwd_ctas * nparam, 32);
  w.flat = p; p += align_up(nparam, 32);
  w.scratch = p;
  w.scratch_doubles = avail - need;
  return MCP_OK;
}

static int check_rollout(const McpRollout* r) {
  MCP_CHECK_ARG(r != nullptr, "null rollout descriptor");
  const McpModel& m = r->model;
  const McpPolicy& p = r->policy;
  MCP_CHECK_ARG(r->M >= 1 && r->H >= 1, "rollout: M=%d H=%d", r->M, r->H);
  MCP_CHECK_ARG(m.Ds >= 1 && m.Ds <= MCP_MAX_DS && m.Du >= 1 && m.Du <= MCP_MAX_DU && m.E >= 1 && m.E <= MCP_MAX_E &&
                    m.D >= 1 && m.D <= MCP_MAX_D, "rollout: model dims out of range (Ds=%d Du=%d E=%d D=%d)", m.Ds, m.Du, m.E, m.D);
  int dfeat = m.use_trig ? m.n_na + 2 * m.n_a + m.Du : m.Ds + m.Du;
  MCP_CHECK_ARG(dfeat == m.D, "rollout: gp-input dimension %d does not match the feature map (%d)", m.D, dfeat);
  MCP_CHECK_ARG(m.kind == 1 || m.E == m.Ds, "rollout: delta-state model needs E == Ds");
  MCP_CHECK_ARG(p.nb >= 1 && p.nb <= 512 && p.Dp >= 1 && p.Dp <= MCP_MAX_DP && p.Du == m.Du && p.Ds == m.Ds,
                "rollout: policy dims out of range (nb=%d Dp=%d Du=%d Ds=%d)", p.nb, p.Dp, p.Du, p.Ds);
  int dp = p.kind == 1 ? p.n_na + 2 * p.n_a : (p.kind == 2 ? 2 * p.Ds : p.Ds);
  MCP_CHECK_ARG(dp == p.Dp, "rollout: policy feature dimension %d does not match kind %d (%d)", p.Dp, p.kind, dp);
  MCP_CHECK_ARG(p.log_ls && p.centers && p.W && (!p.has_bias || p.bias) && (p.kind != 2 || p.target_traj), "rollout: null policy tensor");
  MCP_CHECK_ARG(r->gps && r->x0 && r->states && r->inputs, "rollout: null tensor");
  MCP_CHECK_ARG(!r->need_grad || r->H == 1 || r->jac, "rollout: need_grad requires the jac checkpoint buffer");
  MCP_CHECK_ARG(!r->meas.enabled || r->pol_in, "rollout: the measurement model needs pol_in");
  MCP_CHECK_ARG(r->cost.kind == 0 || r->costs, "rollout: fused cost needs the costs buffer");
  MCP_CHECK_ARG(r->cost.kind != 2 || r->cost.target_traj, "rollout: trajectory cost needs target_traj");
  MCP_CHECK_ARG(r->noise.p_dropout >= 0.0 && r->noise.p_dropout < 1.0, "rollout: p_dropout outside [0,1)");
  for (int e = 0; e < m.E; e++) MCP_CHECK_ARG(r->gps[e].spec.D == m.D, "rollout: gp %d input dim %d != %d", e, r->gps[e].spec.D, m.D);
  return MCP_OK;
}

// argument checks shared by the stand-alone policy forward and backward
static int check_policy_call(const McpPolicy* policy, int M, double p_dropout, const char* fn) {
  MCP_CHECK_ARG(policy != nullptr && M >= 0, "%s: null policy", fn);
  const McpPolicy& p = *policy;
  MCP_CHECK_ARG(p.nb >= 1 && p.nb <= 512 && p.Dp >= 1 && p.Dp <= MCP_MAX_DP && p.Du >= 1 && p.Du <= MCP_MAX_DU && p.Ds >= 1 && p.Ds <= MCP_MAX_DS,
                "%s: policy dims out of range (nb=%d Dp=%d Du=%d Ds=%d)", fn, p.nb, p.Dp, p.Du, p.Ds);
  int dp = p.kind == 1 ? p.n_na + 2 * p.n_a : (p.kind == 2 ? 2 * p.Ds : p.Ds);
  MCP_CHECK_ARG(dp == p.Dp, "%s: feature dimension %d does not match kind %d (%d)", fn, p.Dp, p.kind, dp);
  MCP_CHECK_ARG(p.log_ls && p.centers && p.W && (!p.has_bias || p.bias) && (p.kind != 2 || p.target_traj), "%s: null policy tensor", fn);
  MCP_CHECK_ARG(p_dropout >= 0.0 && p_dropout < 1.0, "%s: p_dropout outside [0,1)", fn);
  return MCP_OK;
}

static int policy_bwd_threads(int nb) { return (nb + 31) / 32 * 32; }

// CTAs of the policy backward: about 1024 resident threads per SM, at most one CTA per particle
static int policy_bwd_ctas(int M, int nb) {
  int sms = 148;
  int dev = 0;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  int per_sm = 1024 / policy_bwd_threads(nb);
  per_sm = per_sm < 1 ? 1 : (per_sm > 8 ? 8 : per_sm);
  const int g = sms * per_sm;
  return M < g ? M : g;
}

}  // namespace mcp

using namespace mcp;

extern "C" __attribute__((visibility("default"))) size_t mcpilco_rollout_workspace_bytes(int M, int H, int E, int D, int Nmax, int nb, int Dp, int Du) {
  size_t fixed = fixed_doubles(M, H, E, D, nb, Dp, Du, E, bwd_grid(M)) * sizeof(double);
  // small rollouts run their E per-output chains concurrently: one K*/V scratch per output
  const size_t copies = ((size_t)M * (size_t)(Nmax > 0 ? Nmax : 1) <= ((size_t)1 << 22)) ? (size_t)(E > 0 ? E : 1) : 1;
  return fixed + copies * mcpilco_gp_predict_workspace_bytes(M, Nmax) + 16384 + 65536;  // + device table of the fused small path
}

extern "C" __attribute__((visibility("default"))) int mcpilco_rollout_fwd(const McpRollout* r, void* stream) {
  if (int e = check_rollout(r)) return e;
  cudaStream_t st = (cudaStream_t)stream;
  Workspace w;
  if (int e = carve(r, w)) return e;
  const int M = r->M, H = r->H, Ds = r->model.Ds, Du = r->model.Du, E = r->model.E, D = r->model.D;
  const bool meas = r->meas.enabled != 0;
  const int Mg = r->M_global > 0 ? r->M_global : M;
  // fan the per-output chains out over side streams when one chain cannot fill the GPU and every output gets a full-M scratch
  int nmax = 1;
  for (int e = 0; e < E; e++) nmax = r->gps[e].N > nmax ? r->gps[e].N : nmax;
  const size_t per_gp = (w.scratch_doubles / (size_t)E) & ~(size_t)31;
  const size_t need_gp = 2 * (size_t)M * (size_t)((nmax + 15) / 16 * 16);
  Fan* fan = (E > 1 && (size_t)M * nmax <= ((size_t)1 << 22) && per_gp >= need_gp) ? get_fan(st) : nullptr;
  MCP_CUDA(cudaMemcpyAsync(r->states, r->x0, sizeof(double) * (size_t)M * Ds, cudaMemcpyDeviceToDevice, st));
  if (meas) {
    MCP_CUDA(cudaMemcpyAsync(r->pol_in, r->x0, sizeof(double) * (size_t)M * Ds, cudaMemcpyDeviceToDevice, st));
    init_nv_kernel<<<cdiv(M, 128), 128, 0, st>>>(r->meas, M, Ds, r->x0, w.nv);
    MCP_LAUNCH_CHECK();
  }
  // cart-pole-sized rollouts whose K^-1 fits a cluster's shared memory: ONE persistent kernel for the whole horizon
  const bool persist = persist_path_ok(r) && w.scratch_doubles >= persist_path_doubles(E);
  if (persist) {
    if (int err = rollout_fwd_persist(r, w.nv, w.scratch, w.scratch_doubles, st)) return err;
  }
  const bool small = persist || (small_path_ok(r) && w.scratch_doubles >= small_path_doubles(M, E, nmax));
  if (small && !persist) {
    if (int err = rollout_fwd_small(r, w.Xs, w.nv, w.scratch, w.scratch_doubles, st)) return err;
  }
  // small rollouts with wide gp inputs: all outputs of a step batched into three launches instead of E chains on side streams
  const bool batched = !small && fan != nullptr && gp_posterior_batched_ok(r->gps, E, r->need_grad != 0) &&
                       w.scratch_doubles >= gp_posterior_batched_doubles(M, E, nmax);
  const McpGpDev* tab = nullptr;
  double* bKs = nullptr;
  if (batched) {
    if (int err = gp_posterior_batched_setup(r->gps, E, M, nmax, w.scratch, w.scratch_doubles, &tab, &bKs, st)) return err;
  }
  for (int t = 0; t < H && !small; t++) {
    const double* x_t = r->states + (size_t)t * M * Ds;
    const double* p_t = meas ? r->pol_in + (size_t)t * M * Ds : x_t;
    const bool fused_tail = Mg <= 2048;  // block-per-particle policy: evaluated by the kernel that made x_t (below), except at t = 0
    if (t == 0 || !fused_tail) {
      if (int err = launch_policy(r->policy, r->model, r->noise, M, Mg, t, t, p_t, x_t, r->inputs + (size_t)t * M * Du,
                                  t < H - 1 ? w.Xs : nullptr, st))
        return err;
    }
    if (t == H - 1) break;
    if (batched) {
      if (int err = gp_posterior_batched(tab, E, D, nmax, w.Xs, M, w.mean, w.var, w.jmean, w.jvar, bKs, st)) return err;
    } else if (fan != nullptr) {
      // small problem: the E per-output chains (K* tile -> contraction -> reduce) are independent; run them side by side
      MCP_CUDA(cudaEventRecord(fan->fork, st));
      for (int e = 0; e < E; e++) {
        cudaStream_t se = e == 0 ? st : fan->side[e];
        if (e > 0) MCP_CUDA(cudaStreamWaitEvent(se, fan->fork, 0));
        if (int err = gp_posterior_chunk(r->gps[e], E, e, w.Xs, M, w.mean, w.var, r->need_grad ? w.jmean : nullptr,
                                         r->need_grad ? w.jvar : nullptr, w.scratch + (size_t)e * per_gp, per_gp, se))
          return err;
        if (e > 0) {
          MCP_CUDA(cudaEventRecord(fan->join[e], se));
          MCP_CUDA(cudaStreamWaitEvent(st, fan->join[e], 0));
        }
      }
    } else {
      for (int e = 0; e < E; e++) {
        if (int err = gp_posterior_chunk(r->gps[e], E, e, w.Xs, M, w.mean, w.var, r->need_grad ? w.jmean : nullptr,
                                         r->need_grad ? w.jvar : nullptr, w.scratch, w.scratch_doubles, st))
          return err;
      }
    }
    if (fused_tail)
      integrate_policy_block_kernel<<<M, policy_block_threads(r->policy.nb), 0, st>>>(
          r->model, r->meas, r->noise, r->policy, M, t, x_t, w.mean, w.var, w.jmean, w.jvar, r->states + (size_t)(t + 1) * M * Ds,
          r->need_grad ? r->jac + (size_t)t * M * E * D : nullptr, p_t, meas ? r->pol_in + (size_t)(t + 1) * M * Ds : nullptr, w.nv,
          r->inputs + (size_t)(t + 1) * M * Du, t + 1 < H - 1 ? w.Xs : nullptr);
    else if (M <= 4096)
      integrate_warp_kernel<<<cdiv(M, 8), 256, 0, st>>>(r->model, r->meas, r->noise, M, t, x_t, w.mean, w.var, w.jmean, w.jvar,
                                                        r->states + (size_t)(t + 1) * M * Ds,
                                                        r->need_grad ? r->jac + (size_t)t * M * E * D : nullptr, p_t,
                                                        meas ? r->pol_in + (size_t)(t + 1) * M * Ds : nullptr, w.nv);
    else
      integrate_kernel<<<cdiv(M, 128), 128, 0, st>>>(r->model, r->meas, r->noise, M, t, x_t, w.mean, w.var, w.jmean, w.jvar,
                                                     r->states + (size_t)(t + 1) * M * Ds,
                                                     r->need_grad ? r->jac + (size_t)t * M * E * D : nullptr, p_t,
                                                     meas ? r->pol_in + (size_t)(t + 1) * M * Ds : nullptr, w.nv);
    MCP_LAUNCH_CHECK();
  }
  if (r->cost.kind != 0) {
    size_t n = (size_t)M * H;
    cost_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(r->cost, M, H, Ds, r->states, r->costs);
    MCP_LAUNCH_CHECK();
    double* stats = r->cost_stats ? r->cost_stats : w.stats;  // [H, 2] per-step {mean, M2}: what shards merge across GPUs
    cost_stats_kernel<<<H, 256, 0, st>>>(M, r->costs, stats);
    MCP_LAUNCH_CHECK();
    if (r->cost_out) {
      cost_final_kernel<<<1, 32, 0, st>>>(M, H, stats, r->cost_out);
      MCP_LAUNCH_CHECK();
    }
  }
  return MCP_OK;
}

extern "C" __attribute__((visibility("default"))) int mcpilco_rollout_bwd(const McpRollout* r, const McpRolloutGrad* g, void* stream) {
  if (int e = check_rollout(r)) return e;
  MCP_CHECK_ARG(g != nullptr, "rollout_bwd: null gradient descriptor");
  MCP_CHECK_ARG(r->H == 1 || r->jac, "rollout_bwd: forward was run without need_grad");
  MCP_CHECK_ARG(g->grad_states || g->grad_inputs || r->cost.kind != 0, "rollout_bwd: no grad_states, no grad_inputs and no fused cost");
  cudaStream_t st = (cudaStream_t)stream;
  Workspace w;
  if (int e = carve(r, w)) return e;
  const int nb = r->policy.nb, Dp = r->policy.Dp, Du = r->policy.Du;
  const int nparam = Dp + nb * Dp + Du * nb + Du;
  const int threads = (nb + 31) / 32 * 32 + 32;  // one thread per basis function + the chain warp
  const size_t ring = (size_t)BW_RING * (3 * r->model.Ds + 2 * Du + r->model.E * r->model.D) * sizeof(double);  // <= 37 KB
  const size_t smem_cb = Dp > 16 ? (size_t)Dp * threads * sizeof(double) : 0;   // the widest instance keeps the centres in shared memory
  // up to 224 basis functions: 256 threads and three resident CTAs per SM (the reference's 400 particles are one wave); else 544 threads
#define MCP_BWD_ONE(DPT, DUT, NT, NC)                                                                             \
  do {                                                                                                            \
    static bool cfg_[MCP_MAX_DEVICES] = {};                                                                       \
    MCP_CUDA(ensure_dynamic_smem(cfg_, rollout_bwd_kernel<DPT, DUT, NT, NC>, 200 * 1024));                        \
    rollout_bwd_kernel<DPT, DUT, NT, NC><<<w.bwd_ctas, threads, ring + smem_cb, st>>>(*r, *g, w.partials, g->g_x0); \
  } while (0)
#define MCP_BWD(DPT, DUT)                                       \
  do {                                                          \
    if (threads <= 256) MCP_BWD_ONE(DPT, DUT, 256, 3);          \
    else MCP_BWD_ONE(DPT, DUT, 544, 1);                         \
  } while (0)
  if (Dp <= 8) { if (Du <= 2) MCP_BWD(8, 2); else MCP_BWD(8, 8); }
  else if (Dp <= 16) { if (Du <= 2) MCP_BWD(16, 2); else MCP_BWD(16, 8); }
  else { if (Du <= 2) MCP_BWD(32, 2); else MCP_BWD(32, 8); }
#undef MCP_BWD
#undef MCP_BWD_ONE
  MCP_LAUNCH_CHECK();
  reduce_partials_kernel<<<cdiv(nparam, 128), 128, 0, st>>>(w.partials, w.bwd_ctas, nparam, w.flat);
  MCP_LAUNCH_CHECK();
  scatter_grads_kernel<<<cdiv(nparam, 128), 128, 0, st>>>(w.flat, Dp, nb, Du, g->g_log_ls, g->g_centers, g->g_W, g->g_bias);
  MCP_LAUNCH_CHECK();
  return MCP_OK;
}

extern "C" __attribute__((visibility("default"))) int mcpilco_policy_forward(const McpPolicy* policy, int M, int t, const double* x, double p_dropout,
                                                                              const uint8_t* masks_t, uint64_t seed, uint64_t particle_offset,
                                                                              double* u, void* stream) {
  if (int e = check_policy_call(policy, M, p_dropout, "policy_forward")) return e;
  if (M == 0) return MCP_OK;
  MCP_CHECK_ARG(x && u, "policy_forward: null state / input buffer");
  McpModel mdl{};
  McpNoise nz{};
  nz.masks = masks_t;
  nz.seed = seed;
  nz.particle_offset = particle_offset;
  nz.p_dropout = p_dropout;
  return launch_policy(*policy, mdl, nz, M, M, t, 0, x, x, u, nullptr, (cudaStream_t)stream);
}

extern "C" __attribute__((visibility("default"))) size_t mcpilco_policy_backward_workspace_bytes(int M, int nb, int Dp, int Du) {
  const size_t nparam = (size_t)Dp + (size_t)nb * Dp + (size_t)Du * nb + Du;
  const int ctas = policy_bwd_ctas(M > 0 ? M : 1, nb);
  return (align_up((size_t)ctas * nparam, 32) + nparam) * sizeof(double) + 256;
}

extern "C" __attribute__((visibility("default"))) int mcpilco_policy_backward(const McpPolicy* policy, int M, int t, const double* x, double p_dropout,
                                                                               const uint8_t* masks_t, uint64_t seed, uint64_t particle_offset,
                                                                               const double* g_u, double* g_x, double* g_log_ls, double* g_centers,
                                                                               double* g_W, double* g_bias, void* workspace, size_t workspace_bytes,
                                                                               void* stream) {
  if (int e = check_policy_call(policy, M, p_dropout, "policy_backward")) return e;
  const McpPolicy& p = *policy;
  MCP_CHECK_ARG(g_log_ls && g_centers && g_W && (!p.has_bias || g_bias), "policy_backward: null gradient output");
  cudaStream_t st = (cudaStream_t)stream;
  const int nb = p.nb, Dp = p.Dp, Du = p.Du;
  if (M == 0) {
    MCP_CUDA(cudaMemsetAsync(g_log_ls, 0, sizeof(double) * Dp, st));
    MCP_CUDA(cudaMemsetAsync(g_centers, 0, sizeof(double) * (size_t)nb * Dp, st));
    MCP_CUDA(cudaMemsetAsync(g_W, 0, sizeof(double) * (size_t)Du * nb, st));
    if (p.has_bias) MCP_CUDA(cudaMemsetAsync(g_bias, 0, sizeof(double) * Du, st));
    return MCP_OK;
  }
  MCP_CHECK_ARG(x && g_u, "policy_backward: null state / gradient buffer");
  MCP_CHECK_ARG(workspace && workspace_bytes >= mcpilco_policy_backward_workspace_bytes(M, nb, Dp, Du), "policy_backward: workspace too small");
  const int nparam = Dp + nb * Dp + Du * nb + Du;
  const int ctas = policy_bwd_ctas(M, nb), threads = policy_bwd_threads(nb);
  double* partials = (double*)align_up((size_t)workspace, 256);
  double* flat = partials + align_up((size_t)ctas * nparam, 32);
  McpNoise nz{};
  nz.masks = masks_t;
  nz.seed = seed;
  nz.particle_offset = particle_offset;
  nz.p_dropout = p_dropout;
  const size_t smem = (size_t)(Dp + Du) * threads * sizeof(double);  // <= 160 KB
#define MCP_PBWD(DPT, DUT)                                                                              \
  do {                                                                                                  \
    static bool cfg_[MCP_MAX_DEVICES] = {};                                                             \
    MCP_CUDA(ensure_dynamic_smem(cfg_, policy_bwd_kernel<DPT, DUT>, 160 * 1024));                       \
    policy_bwd_kernel<DPT, DUT><<<ctas, threads, smem, st>>>(p, nz, M, t, x, g_u, g_x, partials);       \
  } while (0)
  if (Dp <= 8) { if (Du <= 2) MCP_PBWD(8, 2); else MCP_PBWD(8, 8); }
  else if (Dp <= 16) { if (Du <= 2) MCP_PBWD(16, 2); else MCP_PBWD(16, 8); }
  else { if (Du <= 2) MCP_PBWD(32, 2); else MCP_PBWD(32, 8); }
#undef MCP_PBWD
  MCP_LAUNCH_CHECK();
  reduce_partials_kernel<<<cdiv(nparam, 128), 128, 0, st>>>(partials, ctas, nparam, flat);
  MCP_LAUNCH_CHECK();
  scatter_grads_kernel<<<cdiv(nparam, 128), 128, 0, st>>>(flat, Dp, nb, Du, g_log_ls, g_centers, g_W, p.has_bias ? g_bias : nullptr);
  MCP_LAUNCH_CHECK();
  return MCP_OK;
}

extern "C" __attribute__((visibility("default"))) int mcpilco_init_particles(int kind, const double* a, const double* b, int n_modes, int M, int Ds,
                                                                              uint64_t seed, uint64_t particle_offset, const uint64_t* seed_dev, double* x0,
                                                                              void* stream) {
  MCP_CHECK_ARG((kind == 0 || kind == 1) && a && b && n_modes >= 1 && M >= 0 && Ds >= 1 && Ds <= MCP_MAX_DS && (kind == 0 || n_modes == 1),
                "init_particles: bad arguments (kind=%d n_modes=%d M=%d Ds=%d)", kind, n_modes, M, Ds);
  if (M == 0) return MCP_OK;
  MCP_CHECK_ARG(x0 != nullptr, "init_particles: null output");
  init_particles_kernel<<<cdiv(M, 128), 128, 0, (cudaStream_t)stream>>>(kind, a, b, n_modes, M, Ds, seed, particle_offset, seed_dev, x0);
  MCP_LAUNCH_CHECK();
  return MCP_OK;
}
