// K9: exact posterior draws of whole MJP histories on a tree (stochastic mapping), one thread per
// (chain, site) trajectory, written in the trajectory layout of the Rao-Teh sweeps (K6,
// rt_raoteh.cu), so a chain started from a draw needs no burn-in.
//
// Replaces the reference's arbitrary initial history
//   _sampler.get_restricted_feasible_history     raoteh/sampler/_sampler.py:563-643
// by a draw from the posterior itself:
//   node states  FFBS on the tree: x_root ~ pi * L_root, then x_c ~ P_c[x_a, :] * L_c top-down
//                (_sample_mc0.resample_states, raoteh/sampler/_sample_mc0.py:20-93) from the
//                partials rt_prune_loglik stored;
//   branch paths the path on branch c given (x_a, x_c, t_c) by uniformization (Hobolth & Stone
//                2009, section 2.4): with mu = max_s q_s and B = I + Q/mu,
//                  Pr(N = n) ~ Pois(n; mu t_c) (B^n)[x_a, x_c],
//                  Pr(x_i = s) ~ B[x_{i-1}, s] (B^{N-i})[s, x_c],
//                event times = order statistics of N uniforms on (0, t_c); only the events
//                where the state changes are kept.
//
// The program is walked backwards (parents before children), as the DOWN pass of a sweep does,
// and the jumps are written from `cap` downwards with times increasing along each edge: that is
// the upward-program order, child end first, the sweeps read.  Everything is drawn in one
// top-down pass, so the kernel needs no per-trajectory scratch.
#include "rt_common.cuh"
#include "rt_philox.cuh"
#include "../../include/rt_b200.h"

namespace {

constexpr int kBlock = 128;
// longest power table: B^0 .. B^kMaxPow.  The Poisson tail beyond n at rate lambda is below 1e-17
// for n ~ lambda + 9 sqrt(lambda) + 20, so 320 covers mu * t up to ~200 -- about the 255 real jumps
// per branch the uint8 counts hold.  A longer branch falls short of P and gets status 3.
constexpr int kMaxPow = 320;
constexpr double kTailEps = 1e-17;
// header of the workspace: mu, n_pow, then the transposed powers Bt[m][j][i] = (B^m)[i][j]
constexpr int kHeader = 2;

template <int S, int OBS>
__device__ __forceinline__ void load_obs_vec(const void* obs, int slot, int64_t obs_stride,
                                             int64_t site, double (&v)[S]) {
  if (OBS == OBS_CODES) {
    const int k = reinterpret_cast<const uint8_t*>(obs)[(int64_t)slot * obs_stride + site];
#pragma unroll
    for (int s = 0; s < S; ++s) v[s] = (k == RT_MISSING || k == s) ? 1.0 : 0.0;
  } else {
    const unsigned long long mk =
        reinterpret_cast<const unsigned long long*>(obs)[(int64_t)slot * obs_stride + site];
#pragma unroll
    for (int s = 0; s < S; ++s) v[s] = ((mk >> s) & 1ull) ? 1.0 : 0.0;
  }
}

// index of the category u falls in, w >= 0 with total tot > 0 (the sweeps' rule: first s with
// x <= cumulative weight; rounding past the end picks the last positive weight)
template <int S>
__device__ __forceinline__ int draw_categorical(const double (&w)[S], double tot, uint32_t u) {
  const double x = ((double)u + 0.5) * 2.3283064365386963e-10 * tot;
  double cum = 0.0;
  int pick = -1;
#pragma unroll
  for (int s = 0; s < S; ++s) {
    cum += w[s];
    if (pick < 0 && w[s] > 0.0 && x <= cum) pick = s;
  }
  if (pick < 0) {
#pragma unroll
    for (int s = 0; s < S; ++s) if (w[s] > 0.0) pick = s;
  }
  return pick;
}

template <typename TT> __device__ __forceinline__ TT next_up(TT x);
template <> __device__ __forceinline__ float next_up(float x) { return nextafterf(x, INFINITY); }
template <> __device__ __forceinline__ double next_up(double x) { return nextafter(x, (double)INFINITY); }
template <typename TT> __device__ __forceinline__ TT next_down(TT x);
template <> __device__ __forceinline__ float next_down(float x) { return nextafterf(x, 0.0f); }
template <> __device__ __forceinline__ double next_down(double x) { return nextafter(x, 0.0); }

// One block: mu = max_s q_s (1 if Q is zero), n_pow from the Poisson tail at mu * max_b t_b
// (capped at kMaxPow), then Bt[m] = (B^m)^T for m = 0..n_pow.
template <int S>
__device__ __forceinline__ void power_table(const double* __restrict__ Q, const double* __restrict__ length,
                                            int n_nodes, double* __restrict__ ws) {
  __shared__ double B_s[S * S], cur[S * S];
  __shared__ int n_pow_s;
  __shared__ double mu_s;
  const int tid = threadIdx.x;
  if (tid == 0) {
    double mu = 0.0;
    for (int s = 0; s < S; ++s) mu = fmax(mu, -Q[s * S + s]);
    if (!(mu > 0.0)) mu = 1.0;      // B = I: events never change the state
    double tmax = 0.0;
    for (int b = 1; b < n_nodes; ++b) tmax = fmax(tmax, length[b]);
    const double lam = mu * tmax;
    // smallest n >= lam with Pr(N > n) <= p_n r / (1 - r) < kTailEps, r = lam / (n + 1)
    int n = (int)ceil(lam);
    while (n < kMaxPow) {
      const double r = lam / (n + 1);
      const double logp = lam > 0.0 ? -lam + n * log(lam) - lgamma((double)n + 1.0) : (n == 0 ? 0.0 : -INFINITY);
      if (r < 1.0 && exp(logp) * r / (1.0 - r) < kTailEps) break;
      ++n;
    }
    if (n < 2 * S + 8) n = 2 * S + 8;   // paths that need several jumps on a short branch
    if (n > kMaxPow) n = kMaxPow;
    n_pow_s = n;
    mu_s = mu;
    ws[0] = mu;
    ws[1] = (double)n;
  }
  __syncthreads();
  const double mu = mu_s;
  const int n_pow = n_pow_s;
  const int i = tid / S, j = tid % S;
  if (tid < S * S) {
    B_s[tid] = (i == j ? 1.0 : 0.0) + Q[tid] / mu;
    cur[tid] = (i == j) ? 1.0 : 0.0;
  }
  __syncthreads();
  double* Bt = ws + kHeader;
  for (int m = 0; m <= n_pow; ++m) {
    double v = 0.0;
    if (tid < S * S) {
      v = cur[i * S + j];
      Bt[(size_t)m * S * S + j * S + i] = v;
      double nx = 0.0;
#pragma unroll
      for (int l = 0; l < S; ++l) nx = fma(cur[i * S + l], B_s[l * S + j], nx);
      v = nx;
    }
    __syncthreads();
    if (tid < S * S) cur[tid] = v;
    __syncthreads();
  }
}

template <int S>
__global__ void power_table_kernel(const double* __restrict__ Q, const double* __restrict__ length,
                                   int n_nodes, double* __restrict__ ws) {
  power_table<S>(Q, length, n_nodes, ws);
}

// doubles of one power table in the workspace
template <int S>
constexpr size_t table_size() { return kHeader + (size_t)(kMaxPow + 1) * S * S; }

// block c: the table of class c, generator Q + c S^2, at ws + c * table_size
template <int S>
__global__ void power_table_classes_kernel(const double* __restrict__ Q, const double* __restrict__ length,
                                           int n_nodes, double* __restrict__ ws) {
  power_table<S>(Q + (size_t)blockIdx.x * S * S, length, n_nodes, ws + blockIdx.x * table_size<S>());
}

template <typename TT>
struct DrawArgs {
  int n_nodes, n_ops, cap;
  int64_t n_traj, stride, n_sites, traj0, obs_stride, site_stride;
  uint64_t seed;
  long long k;
  const int4* program;
  const int32_t* parent;
  const double* length;
  const double* P;          // [n_nodes][S][S]
  const double* root_distn;
  const void* obs;
  const double* partials;   // [n_store][S][site_stride]
  const int8_t* site_status;
  const double* ws;         // mu, n_pow, Bt[0..n_pow]
  uint8_t* node_state;
  TT* ev_time;
  uint8_t* ev_sb;
  uint8_t* ev_count;
  int32_t* ev_total;
  int32_t* sweep_count;
  double* dwell_sum;
  double* trans_sum;
  int8_t* status;
};

// the site-class mixture's additions (posterior_draw_mixture_kernel): P, partials, power tables
// and statistics are per class, the class drawn per trajectory from class_post [K][stride]
struct MixArgs {
  int K;
  int64_t partials_class_stride, class_post_stride;
  const double* class_post;
  uint8_t* site_class;
};

// p + off for the mixture kernel's per-class inputs; the single-class kernel's pointer untouched
template <bool MIX>
__device__ __forceinline__ const double* at_class(const double* p, size_t off) {
  if constexpr (MIX) return p + off;
  else return p;
}

// class ~ w[k * stride], k < K: draw_categorical's rule; -1 if every weight is 0
__device__ __forceinline__ int draw_class(const double* w, int64_t stride, int K, uint32_t u) {
  double tot = 0.0;
  for (int k = 0; k < K; ++k) tot += w[k * stride];
  if (!(tot > 0.0)) return -1;
  const double x = ((double)u + 0.5) * 2.3283064365386963e-10 * tot;
  double cum = 0.0;
  int last = -1;
  for (int k = 0; k < K; ++k) {
    const double wk = w[k * stride];
    cum += wk;
    if (wk > 0.0) {
      last = k;
      if (x <= cum) break;
    }
  }
  return last;
}

template <int S, int OBS, bool STATS, typename TT>
__global__ void __launch_bounds__(kBlock, 4)
posterior_draw_kernel(DrawArgs<TT> A) {
  constexpr bool MIX = false;
  [[maybe_unused]] const MixArgs X{};
#include "rt_posterior_draw_walk.cuh"
}

template <int S, int OBS, bool STATS, typename TT>
__global__ void __launch_bounds__(kBlock, 4)
posterior_draw_mixture_kernel(DrawArgs<TT> A, MixArgs X) {
  constexpr bool MIX = true;
#include "rt_posterior_draw_walk.cuh"
}

template <int S, int OBS, bool MIX, typename TT>
int launch(const DrawArgs<TT>& A, const MixArgs& X, bool stats, cudaStream_t stream) {
  const size_t smem = sizeof(int4) * A.n_ops + sizeof(double) * (S * S + S + A.n_nodes) +
                      (stats ? sizeof(double) * S * kBlock + sizeof(uint32_t) * S * S * kBlock : 0) +
                      sizeof(int) * A.n_nodes + (MIX ? sizeof(uint32_t) * 8 + kBlock : 0) + 16;
  if (smem > 200 * 1024) return RT_ERR_UNSUPPORTED;
  const unsigned grid = (unsigned)((A.n_traj + kBlock - 1) / kBlock);
  auto go = [&](auto kern, auto... extra) -> int {
    RT_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, kBlock, smem, stream>>>(A, extra...);
    return RT_OK;
  };
  int rc;
  if constexpr (MIX)
    rc = stats ? go(posterior_draw_mixture_kernel<S, OBS, true, TT>, X)
               : go(posterior_draw_mixture_kernel<S, OBS, false, TT>, X);
  else
    rc = stats ? go(posterior_draw_kernel<S, OBS, true, TT>) : go(posterior_draw_kernel<S, OBS, false, TT>);
  if (rc != RT_OK) return rc;
  RT_CUDA_CHECK(cudaGetLastError());
  return RT_OK;
}

// K = 0: rt_posterior_draw (one power table from Q); K >= 1: the mixture (K tables, one block each)
template <int S, typename TT>
int launch_s(const rt_posterior_draw_args& R, const MixArgs& X, const double* ws, cudaStream_t stream) {
  DrawArgs<TT> A;
  A.n_nodes = R.n_nodes; A.n_ops = R.n_ops; A.cap = R.cap;
  A.n_traj = R.n_traj; A.stride = R.traj_stride; A.n_sites = R.n_sites; A.traj0 = R.traj0;
  A.obs_stride = R.obs_stride; A.site_stride = R.site_stride;
  A.seed = R.seed; A.k = R.k;
  A.program = reinterpret_cast<const int4*>(R.program);
  A.parent = R.parent; A.length = R.length; A.P = R.P; A.root_distn = R.root_distn; A.obs = R.obs;
  A.partials = R.partials; A.site_status = R.site_status; A.ws = ws;
  A.node_state = R.node_state; A.ev_time = reinterpret_cast<TT*>(R.ev_time); A.ev_sb = R.ev_sb;
  A.ev_count = R.ev_count; A.ev_total = R.ev_total; A.sweep_count = R.sweep_count;
  A.dwell_sum = R.dwell_sum; A.trans_sum = R.trans_sum; A.status = R.status;
  const bool stats = R.dwell_sum != nullptr && R.trans_sum != nullptr;
  if (X.K == 0) {
    power_table_kernel<S><<<1, 64, 0, stream>>>(R.Q, R.length, R.n_nodes, const_cast<double*>(ws));
    RT_CUDA_CHECK(cudaGetLastError());
    if (R.obs_kind == OBS_CODES) return launch<S, OBS_CODES, false, TT>(A, X, stats, stream);
    return launch<S, OBS_MASK, false, TT>(A, X, stats, stream);
  }
  power_table_classes_kernel<S><<<X.K, 64, 0, stream>>>(R.Q, R.length, R.n_nodes, const_cast<double*>(ws));
  RT_CUDA_CHECK(cudaGetLastError());
  if (R.obs_kind == OBS_CODES) return launch<S, OBS_CODES, true, TT>(A, X, stats, stream);
  return launch<S, OBS_MASK, true, TT>(A, X, stats, stream);
}

template <int S>
int dispatch_s(const rt_posterior_draw_args& R, const MixArgs& X, const double* ws, cudaStream_t stream) {
  if (R.time_f64) {
    if constexpr (S == 7) return RT_ERR_UNSUPPORTED;
    else return launch_s<S, double>(R, X, ws, stream);
  }
  return launch_s<S, float>(R, X, ws, stream);
}

int draw_dispatch(const rt_posterior_draw_args& R, const MixArgs& X, cudaStream_t stream) {
  const int S = R.S;
  double* ws = nullptr;
  const size_t bytes = sizeof(double) * (X.K > 0 ? X.K : 1) * (kHeader + (size_t)(kMaxPow + 1) * S * S);
  RT_CUDA_CHECK(rt_ws_alloc((void**)&ws, bytes, stream));
  int rc;
  switch (S) {
    case 2: rc = dispatch_s<2>(R, X, ws, stream); break;
    case 3: rc = dispatch_s<3>(R, X, ws, stream); break;
    case 4: rc = dispatch_s<4>(R, X, ws, stream); break;
    case 5: rc = dispatch_s<5>(R, X, ws, stream); break;
    case 6: rc = dispatch_s<6>(R, X, ws, stream); break;
    case 7: rc = dispatch_s<7>(R, X, ws, stream); break;
    case 8: rc = dispatch_s<8>(R, X, ws, stream); break;
    default: rc = RT_ERR_UNSUPPORTED;
  }
  rt_ws_free(ws, stream);
  return rc;
}

}  // namespace

int rt_posterior_draw_dispatch(const rt_posterior_draw_args& R, cudaStream_t stream) {
  return draw_dispatch(R, MixArgs{}, stream);
}

int rt_posterior_draw_mixture_dispatch(const rt_posterior_draw_mixture_args& M, cudaStream_t stream) {
  MixArgs X;
  X.K = M.K;
  X.partials_class_stride = M.partials_class_stride;
  X.class_post_stride = M.class_post_stride;
  X.class_post = M.class_post;
  X.site_class = M.site_class;
  return draw_dispatch(M.base, X, stream);
}
