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
__global__ void power_table_kernel(const double* __restrict__ Q, const double* __restrict__ length,
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

template <int S, int OBS, bool STATS, typename TT>
__global__ void __launch_bounds__(kBlock, 4)
posterior_draw_kernel(DrawArgs<TT> A) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  int4* prog_s = reinterpret_cast<int4*>(smem_raw);
  double* B_s = reinterpret_cast<double*>(prog_s + A.n_ops);          // [S][S]
  double* pi_s = B_s + S * S;                                          // [S]
  double* len_s = pi_s + S;                                            // [n_nodes]
  double* dwell_s = len_s + A.n_nodes;                                 // [S][kBlock]
  uint32_t* trans_s = reinterpret_cast<uint32_t*>(dwell_s + (STATS ? S * kBlock : 0));   // [S*S][kBlock]
  int* par_s = reinterpret_cast<int*>(trans_s + (STATS ? S * S * kBlock : 0));           // [n_nodes]
  __shared__ double red[kBlock / 32][S * S + S];

  const int tid = threadIdx.x;
  const double mu = A.ws[0];
  const int n_pow = (int)A.ws[1];
  const double* Bt = A.ws + kHeader;
  for (int i = tid; i < A.n_ops; i += kBlock) prog_s[i] = A.program[i];
  for (int i = tid; i < S * S; i += kBlock) B_s[i] = Bt[S * S + (i % S) * S + i / S];
  if (tid < S) pi_s[tid] = A.root_distn ? A.root_distn[tid] : 1.0;
  for (int i = tid; i < A.n_nodes; i += kBlock) { len_s[i] = A.length[i]; par_s[i] = A.parent[i]; }
  if (STATS) {
#pragma unroll
    for (int s = 0; s < S; ++s) dwell_s[s * kBlock + tid] = 0.0;
#pragma unroll
    for (int q = 0; q < S * S; ++q) trans_s[q * kBlock + tid] = 0u;
  }
  __syncthreads();

  const int64_t traj = (int64_t)blockIdx.x * kBlock + tid;
  const int64_t site = traj < A.n_traj ? (A.traj0 + traj) % A.n_sites : 0;
  bool active = traj < A.n_traj && A.status[traj] == RT_SITE_OK;
  if (active && A.site_status && A.site_status[site] != RT_SITE_OK) {
    A.status[traj] = A.site_status[site];
    active = false;
  }

  if (active) {
    const int64_t st = A.stride;
    uint8_t* ns_p = A.node_state + traj;
    uint8_t* cnt_p = A.ev_count + traj;
    TT* evt_p = A.ev_time + (size_t)traj * A.cap;
    uint8_t* evs_p = A.ev_sb + (size_t)traj * A.cap;
    Philox rng;
    rng.init(A.seed, (uint64_t)(A.traj0 + traj), (uint32_t)A.k);
    // substream 1: the draw's own words (a sweep uses substream 0); word 0 draws the root, words
    // 2 and 3 seed the PCG32 stream of everything else, as in the sweeps
    rng.block(1u, 0u);
    uint64_t pcg_state = ((uint64_t)rng.out[3] << 32) | (uint64_t)rng.out[2];
    const uint64_t pcg_inc = ((uint64_t)(A.traj0 + traj) << 1) | 1ull;
    auto pcg_next = [&]() -> uint32_t {
      const uint64_t old = pcg_state;
      pcg_state = old * 6364136223846793005ull + pcg_inc;
      const uint32_t xs = (uint32_t)(((old >> 18) ^ old) >> 27);
      const uint32_t rot = (uint32_t)(old >> 59);
      return (xs >> rot) | (xs << ((32u - rot) & 31u));
    };
    pcg_next();
    auto unit = [&]() -> double { return ((double)pcg_next() + 0.5) * 2.3283064365386963e-10; };

    int8_t fail = RT_SITE_OK;
    // ---- root ~ pi * L_root (store index of the OP_ROOT op) ----
    {
      const int4 op = prog_s[A.n_ops - 1];
      const double* Lp = A.partials + (int64_t)op.w * S * A.site_stride + site;
      double w[S], tot = 0.0;
#pragma unroll
      for (int s = 0; s < S; ++s) { w[s] = pi_s[s] * Lp[(int64_t)s * A.site_stride]; tot += w[s]; }
      if (!(tot > 0.0)) fail = RT_SITE_STRUCTURAL_ZERO;
      else ns_p[(int64_t)op.y * st] = (uint8_t)draw_categorical<S>(w, tot, rng.out[0]);
    }
    int wr = A.cap;
    for (int ip = A.n_ops - 1; ip >= 0 && fail == RT_SITE_OK; --ip) {
      const int4 op = prog_s[ip];
      const int code = op.x & 0xff;
      if (code > OP_MSG_ONES) continue;
      const int c = op.y;
      const int xa = ns_p[(int64_t)par_s[c] * st];
      // ---- node state: x_c ~ P_c[x_a, :] * L_c ----
      double L[S];
      if (code == OP_MSG_SLOT) {
        const double* Lp = A.partials + (int64_t)op.w * S * A.site_stride + site;
#pragma unroll
        for (int s = 0; s < S; ++s) L[s] = Lp[(int64_t)s * A.site_stride];
      } else if (code == OP_MSG_OBS) {
        load_obs_vec<S, OBS>(A.obs, op.z, A.obs_stride, site, L);
      } else {
#pragma unroll
        for (int s = 0; s < S; ++s) L[s] = 1.0;
      }
      const double* Prow = A.P + ((size_t)c * S + xa) * S;
      double w[S], tot = 0.0;
#pragma unroll
      for (int s = 0; s < S; ++s) { w[s] = __ldg(Prow + s) * L[s]; tot += w[s]; }
      if (!(tot > 0.0)) { fail = RT_SITE_STRUCTURAL_ZERO; break; }
      const int xc = draw_categorical<S>(w, tot, pcg_next());
      ns_p[(int64_t)c * st] = (uint8_t)xc;

      // ---- path on the branch given (x_a, x_c, t_c) ----
      const double tc = len_s[c];
      int kept = 0;
      int x = xa;
      TT prev = (TT)0;
      if (tc > 0.0) {
        // largest stored time: the largest TT value below t_c
        TT hi = (TT)tc;
        if (!((double)hi < tc)) hi = next_down(hi);
        const double lam = mu * tc;
        const double* Btc = Bt + (size_t)xc * S;          // Bt[m][xc][s] = (B^m)[s][xc]
        // Pr(N = n) ~ Pois(n; lam) (B^n)[xa, xc]: sum of the series up to n_pow, or until the
        // Poisson tail cannot move it (for n > lam the tail is below p_n r / (1 - r))
        double p = exp(-lam), tot_n = 0.0;
        int n_end = n_pow;
        for (int n = 0; n <= n_pow; ++n) {
          tot_n = fma(p, __ldg(Btc + (size_t)n * S * S + xa), tot_n);
          const double r = lam / (n + 1);
          if (r < 0.5 && tot_n > 0.0 && p * 2.0 * r < kTailEps * tot_n) { n_end = n; break; }
          p *= r;
        }
        const double pac = __ldg(Prow + xc);
        // truncation guard: the series must reach P_c[xa, xc] (1e-14 absolute: the accuracy of
        // the smallest entries of expm)
        if (!(tot_n > 0.0) || tot_n < pac * (1.0 - 1e-12) - 1e-14) { fail = 3; break; }
        const double xu = unit() * tot_n;
        int N = -1;
        {
          double q = exp(-lam), cum = 0.0;
          int last = 0;            // rounding past the end: the last n of positive weight
          for (int n = 0; n <= n_end; ++n) {
            const double wn = q * __ldg(Btc + (size_t)n * S * S + xa);
            cum += wn;
            if (wn > 0.0) {
              last = n;
              if (xu <= cum) { N = n; break; }
            }
            q *= lam / (n + 1);
          }
          if (N < 0) N = last;
        }
        // events 1..N: state given the previous one and the end state, time as the next order
        // statistic of N uniforms on (0, 1): U_(i) = 1 - (1 - U_(i-1)) V^(1 / (N - i + 1))
        double u_prev = 0.0;
        for (int i = 1; i <= N; ++i) {
          const double v = unit();
          const double u_i = 1.0 - (1.0 - u_prev) * exp(log(v) / (double)(N - i + 1));
          u_prev = u_i;
          int nx = xc;
          if (i < N) {
            const double* Bm = Btc + (size_t)(N - i) * S * S;
            double ws[S], tw = 0.0;
#pragma unroll
            for (int s = 0; s < S; ++s) { ws[s] = B_s[x * S + s] * __ldg(Bm + s); tw += ws[s]; }
            nx = tw > 0.0 ? draw_categorical<S>(ws, tw, pcg_next()) : -1;
            if (nx < 0) { fail = 3; break; }
          }
          if (nx == x) continue;
          // a real jump: stored strictly inside (0, t_c) and after the previous one in TT
          TT tau = (TT)(u_i * tc);
          if (tau > hi) tau = hi;
          if (!(tau > prev)) tau = next_up(prev);
          if (tau > hi) { fail = 3; break; }
          if (STATS) {
            dwell_s[x * kBlock + tid] += (double)(tau - prev);
            trans_s[(x * S + nx) * kBlock + tid] += 1u;
          }
          --wr;
          if (wr >= 0) { evt_p[wr] = tau; evs_p[wr] = (uint8_t)x; }
          prev = tau;
          ++kept;
          x = nx;
        }
        if (fail != RT_SITE_OK) break;
        if (kept > 255) { fail = 3; break; }
      }
      if (STATS) dwell_s[x * kBlock + tid] += tc - (double)prev;
      cnt_p[(int64_t)c * st] = (uint8_t)kept;
    }
    if (fail == RT_SITE_OK && wr < 0) fail = 4;
    if (fail != RT_SITE_OK) {
      A.status[traj] = fail;
      A.ev_total[traj] = 0;
    } else {
      A.ev_total[traj] = A.cap - wr;
      if (A.sweep_count) A.sweep_count[traj] = (int32_t)(A.k + 1);
    }
  }

  if (STATS && A.dwell_sum) {
#pragma unroll
    for (int q = 0; q < S + S * S; ++q) {
      const double mine = q < S ? dwell_s[(q < S ? q : 0) * kBlock + tid]
                                : (double)trans_s[(q >= S ? q - S : 0) * kBlock + tid];
      const double v = rt_warp_sum(mine);
      if ((tid & 31) == 0) red[tid >> 5][q] = v;
    }
    __syncthreads();
    if (tid < S + S * S) {
      double t = 0.0;
      for (int i = 0; i < kBlock / 32; ++i) t += red[i][tid];
      if (t != 0.0) atomicAdd(tid < S ? &A.dwell_sum[tid] : &A.trans_sum[tid - S], t);
    }
  }
}

template <int S, int OBS, typename TT>
int launch(const DrawArgs<TT>& A, bool stats, cudaStream_t stream) {
  const size_t smem = sizeof(int4) * A.n_ops + sizeof(double) * (S * S + S + A.n_nodes) +
                      (stats ? sizeof(double) * S * kBlock + sizeof(uint32_t) * S * S * kBlock : 0) +
                      sizeof(int) * A.n_nodes + 16;
  if (smem > 200 * 1024) return RT_ERR_UNSUPPORTED;
  const unsigned grid = (unsigned)((A.n_traj + kBlock - 1) / kBlock);
  if (stats) {
    auto kern = posterior_draw_kernel<S, OBS, true, TT>;
    RT_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, kBlock, smem, stream>>>(A);
  } else {
    auto kern = posterior_draw_kernel<S, OBS, false, TT>;
    RT_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, kBlock, smem, stream>>>(A);
  }
  RT_CUDA_CHECK(cudaGetLastError());
  return RT_OK;
}

template <int S, typename TT>
int launch_s(const rt_posterior_draw_args& R, const double* ws, cudaStream_t stream) {
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
  power_table_kernel<S><<<1, 64, 0, stream>>>(R.Q, R.length, R.n_nodes, const_cast<double*>(ws));
  RT_CUDA_CHECK(cudaGetLastError());
  if (R.obs_kind == OBS_CODES) return launch<S, OBS_CODES, TT>(A, stats, stream);
  return launch<S, OBS_MASK, TT>(A, stats, stream);
}

template <int S>
int dispatch_s(const rt_posterior_draw_args& R, const double* ws, cudaStream_t stream) {
  if (R.time_f64) {
    if constexpr (S == 7) return RT_ERR_UNSUPPORTED;
    else return launch_s<S, double>(R, ws, stream);
  }
  return launch_s<S, float>(R, ws, stream);
}

}  // namespace

int rt_posterior_draw_dispatch(const rt_posterior_draw_args& R, cudaStream_t stream) {
  const int S = R.S;
  double* ws = nullptr;
  const size_t bytes = sizeof(double) * (kHeader + (size_t)(kMaxPow + 1) * S * S);
  RT_CUDA_CHECK(rt_ws_alloc((void**)&ws, bytes, stream));
  int rc;
  switch (S) {
    case 2: rc = dispatch_s<2>(R, ws, stream); break;
    case 3: rc = dispatch_s<3>(R, ws, stream); break;
    case 4: rc = dispatch_s<4>(R, ws, stream); break;
    case 5: rc = dispatch_s<5>(R, ws, stream); break;
    case 6: rc = dispatch_s<6>(R, ws, stream); break;
    case 7: rc = dispatch_s<7>(R, ws, stream); break;
    case 8: rc = dispatch_s<8>(R, ws, stream); break;
    default: rc = RT_ERR_UNSUPPORTED;
  }
  rt_ws_free(ws, stream);
  return rc;
}
