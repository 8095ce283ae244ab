// K10: forward (prior) simulation of tree MJP sites, one thread per site, under one MJP or a
// site-class mixture, written where the posterior kernels read: leaf codes in the RT_OBS_CODES
// layout of the pruning pass, whole histories in the trajectory layout of the Rao-Teh sweeps (K6).
//
// Replaces the reference's host simulators
//   _sampler.get_forward_sample / gen_forward_samples   raoteh/sampler/_sampler.py:67-235
// (jump by jump, one history per call) and the per-edge expm rows of synth.simulate_leaf_codes.
//
// Every state draw reads one entry of a Walker alias table (Walker 1977; Vose 1991): a setup kernel
// builds one table per sampled row once per call -- the class weights, the root distribution, and
// per class either every (edge, parent state) row of P (NODES) or every row of the jump chain
// Q[s, :] / q_s (HISTORY).  A draw is then O(1) whatever S is, and the walk's registers do not
// depend on S: the tables stay in global memory (L2-resident at the sizes of the library's
// shapes), the program, lengths and the sites' node states in shared memory.
#include "rt_common.cuh"
#include "rt_philox.cuh"
#include "../../include/rt_b200.h"

namespace {

constexpr int kBlock = 128;
// the forward simulation's Philox substream (rt_b200.h): sweeps use 0, the exact draws 1 and 2, the
// warp kernel 0 .. (n_parts + 2)(n_ops + 1) - 1 < 65535
constexpr uint32_t kSubstream = 0xffffu;
// table offsets (entries): the root table, the class table, then the per-class rows
constexpr int kRootOff = 0;
constexpr int kClassOff = 64;
constexpr int kRowsOff = 64 + 256;
// shared-memory budget of the statistics accumulators (all replicas), and the largest single copy
constexpr size_t kStatsBudget = 64 * 1024;
constexpr size_t kStatsMax = 160 * 1024;
constexpr size_t kSmemMax = 200 * 1024;

// Alias table of the row w[0..n) (negative entries and NaN count as 0; entry `skip` is left out,
// -1 = none): entry j = (thr_j << 8) | alias_j with thr_j = floor(2^24 * (probability kept at j)).
// Vose's pairing of small (n w_j / tot < 1) and large entries, run as two forward scans over the
// row with the working values in p[0..n) (processed entries are marked -1), so no work lists are
// needed.  w = NULL is the uniform row; a row without positive weight also draws uniformly.
__device__ void build_alias(const double* w, int n, int skip, double* p, uint32_t* out) {
  double tot = 0.0;
  int any_pos = 0;
  double best = -1.0;
  for (int j = 0; j < n; ++j) {
    const double wj = w ? w[j] : 1.0;
    const double v = (j == skip || !(wj > 0.0)) ? 0.0 : wj;
    p[j] = v;
    tot += v;
    if (v > best) { best = v; any_pos = j; }
  }
  if (!(tot > 0.0)) {
    for (int j = 0; j < n; ++j) out[j] = 0xffffff00u | (uint32_t)j;
    return;
  }
  const double scale = (double)n / tot;
  for (int j = 0; j < n; ++j) p[j] *= scale;
  auto small_from = [&](int i) { while (i < n && !(p[i] >= 0.0 && p[i] < 1.0)) ++i; return i; };
  auto large_from = [&](int i) { while (i < n && !(p[i] >= 1.0)) ++i; return i; };
  int scan = small_from(0);
  int s = scan;
  int l = large_from(0);
  while (s < n && l < n) {
    const double ps = p[s];
    uint32_t thr = (uint32_t)(ps * 16777216.0);
    if (thr > 0xffffffu) thr = 0xffffffu;
    out[s] = (thr << 8) | (uint32_t)l;
    p[s] = -1.0;
    double pl = p[l] - (1.0 - ps);
    if (pl < 0.0) pl = 0.0;
    p[l] = pl;
    if (pl < 1.0) {
      s = l;                      // the large entry turned small: pair it next
      l = large_from(l + 1);
    } else {
      scan = small_from(scan);
      s = scan;
    }
  }
  // left over by rounding: entries of (almost) exactly one column keep their column
  for (int j = 0; j < n; ++j) {
    if (p[j] < 0.0) continue;
    out[j] = p[j] > 0.0 ? (0xffffff00u | (uint32_t)j) : (uint32_t)any_pos;
  }
}

// one draw from an alias table of n entries: column from u1, kept against u2
__device__ __forceinline__ int alias_draw(const uint32_t* __restrict__ tab, int n, uint32_t u1, uint32_t u2) {
  const int j = (int)__umulhi(u1, (uint32_t)n);
  const uint32_t e = __ldg(tab + j);
  return (u2 >> 8) < (e >> 8) ? j : (int)(e & 0xffu);
}

struct SimArgs {
  int S, n_nodes, n_ops, K, cap, n_rep;
  int64_t n_traj, stride, traj0, obs_stride, tmpl_stride, tmpl_n_sites;
  uint64_t seed;
  long long k;
  const int4* program;
  const int32_t* parent;
  const double* length;
  const int32_t* obs_slot;
  const uint8_t* tmpl;
  const uint32_t* tab;       // root, class, per-class rows (kRootOff / kClassOff / kRowsOff)
  const double* inv_rate;    // HISTORY: [K][S] 1 / q_s, 0 where q_s = 0
  uint8_t* obs;
  uint8_t* site_class;
  uint8_t* node_state;
  void* ev_time;
  uint8_t* ev_sb;
  uint8_t* ev_count;
  int32_t* ev_total;
  double* dwell_sum;
  double* trans_sum;
  int8_t* status;
};

// rows: 0 = root distribution (S), 1 = class weights (K), then per class the NODES rows of P
// [K][n_nodes][S] or the HISTORY rows of the jump chain [K][S] (those also write 1 / q_s)
__global__ void build_tables_kernel(int mode, int S, int K, int n_nodes, const double* __restrict__ root_distn,
                                    const double* __restrict__ class_weight, const double* __restrict__ P,
                                    const double* __restrict__ Q, uint32_t* tab, double* inv_rate,
                                    double* scratch, int n_rows) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_rows) return;
  if (r <= 1) {
    const int n = r == 0 ? S : K;
    const int off = r == 0 ? kRootOff : kClassOff;
    const double* w = r == 0 ? root_distn : class_weight;
    build_alias(w, n, -1, scratch + off, tab + off);
    return;
  }
  const size_t row = (size_t)(r - 2);
  const size_t off = kRowsOff + row * S;
  if (mode == RT_SIM_NODES) {
    build_alias(P + row * S, S, -1, scratch + off, tab + off);
  } else {
    const int s = (int)(row % S);
    const double* q = Q + row * S;
    double tot = 0.0;
    for (int j = 0; j < S; ++j)
      if (j != s && q[j] > 0.0) tot += q[j];
    inv_rate[row] = tot > 0.0 ? 1.0 / tot : 0.0;
    build_alias(q, S, s, scratch + off, tab + off);
  }
}

template <typename TT> __device__ __forceinline__ TT next_up(TT x);
template <> __device__ __forceinline__ float next_up(float x) { return nextafterf(x, INFINITY); }
template <> __device__ __forceinline__ double next_up(double x) { return nextafter(x, (double)INFINITY); }
template <typename TT> __device__ __forceinline__ TT next_down(TT x);
template <> __device__ __forceinline__ float next_down(float x) { return nextafterf(x, 0.0f); }
template <> __device__ __forceinline__ double next_down(double x) { return nextafter(x, 0.0); }

template <int MODE, bool STATS, typename TT>
__global__ void __launch_bounds__(kBlock)
forward_kernel(SimArgs A) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int S = A.S, K = A.K, n = A.n_nodes;
  int4* prog_s = reinterpret_cast<int4*>(smem_raw);
  double* len_s = reinterpret_cast<double*>(prog_s + A.n_ops);                  // [n_nodes]
  double* dwell_s = len_s + n;                                                   // [n_rep][K][S]
  int* par_s = reinterpret_cast<int*>(dwell_s + (STATS ? A.n_rep * K * S : 0)); // [n_nodes]
  int* slot_s = par_s + n;                                                       // [n_nodes]
  uint32_t* trans_s = reinterpret_cast<uint32_t*>(slot_s + n);                   // [n_rep][K][S][S]
  uint8_t* ns_s = reinterpret_cast<uint8_t*>(trans_s + (STATS ? A.n_rep * K * S * S : 0));  // [n_nodes][kBlock]

  const int tid = threadIdx.x;
  for (int i = tid; i < A.n_ops; i += kBlock) prog_s[i] = A.program[i];
  for (int i = tid; i < n; i += kBlock) {
    len_s[i] = A.length ? A.length[i] : 0.0;
    par_s[i] = A.parent[i];
    slot_s[i] = A.obs_slot ? A.obs_slot[i] : -1;
  }
  if (STATS) {
    for (int i = tid; i < A.n_rep * K * S; i += kBlock) dwell_s[i] = 0.0;
    for (int i = tid; i < A.n_rep * K * S * S; i += kBlock) trans_s[i] = 0u;
  }
  __syncthreads();
  const int rep = (tid >> 5) % A.n_rep;
  double* dwell_r = dwell_s + (size_t)rep * K * S;
  uint32_t* trans_r = trans_s + (size_t)rep * K * S * S;
  const uint32_t* root_tab = A.tab + kRootOff;
  const uint32_t* class_tab = A.tab + kClassOff;
  const uint32_t* rows = A.tab + kRowsOff;
  uint8_t* my_ns = ns_s + tid;

  for (int64_t t0 = (int64_t)blockIdx.x * kBlock; t0 < A.n_traj; t0 += (int64_t)gridDim.x * kBlock) {
    const int64_t t = t0 + tid;
    if (t >= A.n_traj) continue;
    const uint64_t g = (uint64_t)(A.traj0 + t);
    Philox rng;
    rng.init(A.seed, g, (uint32_t)A.k);
    rng.block(kSubstream, 0u);
    // words 0, 1: the class; words 2, 3 seed the PCG32 stream of every other draw (as the sweeps)
    const int cls = K > 1 ? alias_draw(class_tab, K, rng.out[0], rng.out[1]) : 0;
    if (A.site_class) A.site_class[t] = (uint8_t)cls;
    uint64_t pcg_state = ((uint64_t)rng.out[3] << 32) | (uint64_t)rng.out[2];
    const uint64_t pcg_inc = (g << 1) | 1ull;
    auto pcg_next = [&]() -> uint32_t {
      const uint64_t old = pcg_state;
      pcg_state = old * 6364136223846793005ull + pcg_inc;
      const uint32_t xs = (uint32_t)(((old >> 18) ^ old) >> 27);
      const uint32_t rot = (uint32_t)(old >> 59);
      return (xs >> rot) | (xs << ((32u - rot) & 31u));
    };
    pcg_next();

    // the value written for node v's leaf cell: the state, or RT_MISSING where the template is
    auto emit = [&](int v, int x) {
      my_ns[v * kBlock] = (uint8_t)x;
      if (A.node_state) A.node_state[(int64_t)v * A.stride + t] = (uint8_t)x;
      const int slot = slot_s[v];
      if (slot >= 0 && A.obs) {
        int code = x;
        if (A.tmpl && A.tmpl[(int64_t)slot * A.tmpl_stride + (int64_t)(g % (uint64_t)A.tmpl_n_sites)] == RT_MISSING)
          code = RT_MISSING;
        A.obs[(int64_t)slot * A.obs_stride + t] = (uint8_t)code;
      }
    };
    {
      const uint32_t u1 = pcg_next(), u2 = pcg_next();
      emit(0, alias_draw(root_tab, S, u1, u2));
    }
    const uint32_t* cls_rows = rows + (size_t)cls * (MODE == RT_SIM_NODES ? (size_t)n * S * S : (size_t)S * S);
    [[maybe_unused]] const double* inv_q = A.inv_rate + (size_t)cls * S;
    [[maybe_unused]] TT* evt_p = nullptr;
    [[maybe_unused]] uint8_t* evs_p = nullptr;
    if constexpr (MODE == RT_SIM_HISTORY) {
      evt_p = reinterpret_cast<TT*>(A.ev_time) + (size_t)t * A.cap;
      evs_p = A.ev_sb + (size_t)t * A.cap;
    }
    int wr = A.cap;
    int8_t fail = RT_SITE_OK;
    for (int ip = A.n_ops - 1; ip >= 0; --ip) {
      const int4 op = prog_s[ip];
      if ((op.x & 0xff) > OP_MSG_ONES) continue;
      const int c = op.y;
      const int xa = my_ns[par_s[c] * kBlock];
      int xc;
      if constexpr (MODE == RT_SIM_NODES) {
        const uint32_t u1 = pcg_next(), u2 = pcg_next();
        xc = alias_draw(cls_rows + ((size_t)c * S + xa) * S, S, u1, u2);
      } else {
        // jump by jump: dwell ~ Exp(q_x), next state from the jump chain's row of x
        const double tc = len_s[c];
        TT hi = (TT)tc;                       // largest stored time: the largest TT below t_c
        if (!((double)hi < tc)) hi = next_down(hi);
        double tau_d = 0.0;
        TT prev = (TT)0;
        int x = xa, kept = 0;
        for (;;) {
          const double iq = __ldg(inv_q + x);
          if (!(iq > 0.0)) break;
          const double u = ((double)pcg_next() + 0.5) * 2.3283064365386963e-10;
          tau_d -= log(u) * iq;
          if (!(tau_d < tc)) break;
          const uint32_t u1 = pcg_next(), u2 = pcg_next();
          const int nx = alias_draw(cls_rows + (size_t)x * S, S, u1, u2);
          // stored strictly inside (0, t_c) and after the previous jump in TT
          TT tau = (TT)tau_d;
          if (tau > hi) tau = hi;
          if (!(tau > prev)) tau = next_up(prev);
          if (tau > hi) fail = 3;
          if (STATS) {
            atomicAdd(&dwell_r[cls * S + x], (double)tau - (double)prev);
            atomicAdd(&trans_r[(cls * S + x) * S + nx], 1u);
          }
          --wr;
          if (wr >= 0 && fail == RT_SITE_OK) { evt_p[wr] = tau; evs_p[wr] = (uint8_t)x; }
          prev = tau;
          ++kept;
          x = nx;
        }
        if (kept > 255) fail = 3;
        if (STATS) atomicAdd(&dwell_r[cls * S + x], tc - (double)prev);
        A.ev_count[(int64_t)c * A.stride + t] = (uint8_t)(kept > 255 ? 255 : kept);
        xc = x;
      }
      emit(c, xc);
    }
    if constexpr (MODE == RT_SIM_HISTORY) {
      if (fail == RT_SITE_OK && wr < 0) fail = 4;
      A.status[t] = fail;
      A.ev_total[t] = fail == RT_SITE_OK ? A.cap - wr : 0;
    } else {
      if (A.status) A.status[t] = RT_SITE_OK;
    }
  }

  if (STATS) {
    __syncthreads();
    for (int i = tid; i < K * S; i += kBlock) {
      double v = 0.0;
      for (int r = 0; r < A.n_rep; ++r) v += dwell_s[(size_t)r * K * S + i];
      if (v != 0.0) atomicAdd(&A.dwell_sum[i], v);
    }
    for (int i = tid; i < K * S * S; i += kBlock) {
      uint32_t v = 0;
      for (int r = 0; r < A.n_rep; ++r) v += trans_s[(size_t)r * K * S * S + i];
      if (v) atomicAdd(&A.trans_sum[i], (double)v);
    }
  }
}

template <int MODE, bool STATS, typename TT>
int launch(const SimArgs& A, size_t smem, cudaStream_t stream) {
  auto kern = forward_kernel<MODE, STATS, TT>;
  RT_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int dev = 0, n_sm = 0, per_sm = 0;
  RT_CUDA_CHECK(cudaGetDevice(&dev));
  RT_CUDA_CHECK(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
  RT_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kBlock, smem));
  if (per_sm < 1) return RT_ERR_UNSUPPORTED;
  // a grid of resident blocks walks the sites in strides: the statistics are flushed once a block
  const int64_t need = (A.n_traj + kBlock - 1) / kBlock;
  const int64_t cap_blocks = (int64_t)n_sm * per_sm;
  const unsigned grid = (unsigned)(need < cap_blocks ? need : cap_blocks);
  kern<<<grid, kBlock, smem, stream>>>(A);
  RT_CUDA_CHECK(cudaGetLastError());
  return RT_OK;
}

}  // namespace

int rt_forward_simulate_dispatch(const rt_forward_args& R, cudaStream_t stream) {
  const int S = R.S, K = R.K, n = R.n_nodes;
  const bool hist = R.mode == RT_SIM_HISTORY;
  const bool stats = hist && R.dwell_sum != nullptr;
  const size_t n_rows = hist ? (size_t)K * S : (size_t)K * n * S;
  const size_t n_tab = kRowsOff + n_rows * S;
  // shared memory: program, lengths, parents, leaf slots, the block's node states, statistics
  const size_t per_copy = stats ? (size_t)K * S * sizeof(double) + (size_t)K * S * S * sizeof(uint32_t) : 0;
  if (per_copy > kStatsMax) return RT_ERR_UNSUPPORTED;
  int n_rep = 1;
  if (stats) {
    n_rep = (int)(kStatsBudget / per_copy);
    n_rep = n_rep < 1 ? 1 : (n_rep > kBlock / 32 ? kBlock / 32 : n_rep);
  }
  const size_t smem = sizeof(int4) * R.n_ops + sizeof(double) * n + per_copy * n_rep +
                      2 * sizeof(int) * n + (size_t)n * kBlock;
  if (smem > kSmemMax) return RT_ERR_UNSUPPORTED;

  void* ws = nullptr;
  const size_t tab_bytes = (n_tab * sizeof(uint32_t) + 15) & ~(size_t)15;
  const size_t inv_bytes = hist ? (size_t)K * S * sizeof(double) : 0;
  const size_t scratch_bytes = n_tab * sizeof(double);
  RT_CUDA_CHECK(rt_ws_alloc(&ws, tab_bytes + inv_bytes + scratch_bytes, stream));
  uint32_t* tab = reinterpret_cast<uint32_t*>(ws);
  double* inv_rate = reinterpret_cast<double*>(reinterpret_cast<char*>(ws) + tab_bytes);
  double* scratch = reinterpret_cast<double*>(reinterpret_cast<char*>(ws) + tab_bytes + inv_bytes);
  const int rows_total = (int)(2 + n_rows);
  build_tables_kernel<<<(rows_total + 127) / 128, 128, 0, stream>>>(
      R.mode, S, K, n, R.root_distn, R.class_weight, R.P, R.Q, tab, inv_rate, scratch, rows_total);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    rt_ws_free(ws, stream);
    RT_CUDA_CHECK(e);
  }

  SimArgs A;
  A.S = S; A.n_nodes = n; A.n_ops = R.n_ops; A.K = K; A.cap = R.cap; A.n_rep = n_rep;
  A.n_traj = R.n_traj; A.stride = R.traj_stride; A.traj0 = R.traj0; A.obs_stride = R.obs_stride;
  A.tmpl_stride = R.tmpl_stride; A.tmpl_n_sites = R.tmpl_n_sites;
  A.seed = R.seed; A.k = R.k;
  A.program = reinterpret_cast<const int4*>(R.program);
  A.parent = R.parent; A.length = R.length; A.obs_slot = R.obs_slot; A.tmpl = R.tmpl;
  A.tab = tab; A.inv_rate = inv_rate;
  A.obs = R.obs; A.site_class = R.site_class; A.node_state = R.node_state;
  A.ev_time = R.ev_time; A.ev_sb = R.ev_sb; A.ev_count = R.ev_count; A.ev_total = R.ev_total;
  A.dwell_sum = R.dwell_sum; A.trans_sum = R.trans_sum; A.status = R.status;
  int rc;
  if (!hist) rc = launch<RT_SIM_NODES, false, float>(A, smem, stream);
  else if (R.time_f64) rc = stats ? launch<RT_SIM_HISTORY, true, double>(A, smem, stream)
                                  : launch<RT_SIM_HISTORY, false, double>(A, smem, stream);
  else rc = stats ? launch<RT_SIM_HISTORY, true, float>(A, smem, stream)
                  : launch<RT_SIM_HISTORY, false, float>(A, smem, stream);
  rt_ws_free(ws, stream);
  return rc;
}
