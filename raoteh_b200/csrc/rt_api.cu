// C-ABI entry points of librt_b200.so (see include/rt_b200.h).
#include "rt_common.cuh"
#include "../../include/rt_b200.h"
#include <stdio.h>
#include <string.h>

static thread_local char g_err[512] = "";

void rt_set_last_error(cudaError_t e, const char* file, int line) {
  snprintf(g_err, sizeof(g_err), "CUDA error %d (%s) at %s:%d", (int)e, cudaGetErrorString(e), file, line);
}
// Workspaces come from a private stream-ordered pool per device (cudaMemPoolCreate), so the
// library never touches the attributes of the device's default pool.  Freed blocks stay cached
// in the pool (release threshold = max) until rt_release_workspace() trims it; the largest
// per-call workspaces are bounded by the dispatchers (rt_raoteh.cu launches in trajectory
// chunks, rt_tmjp.cu sizes its scratch by resident warps, not by trajectories).
static cudaMemPool_t g_pool[64] = {};
static cudaError_t ws_pool(cudaMemPool_t* out) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
  if (!g_pool[dev]) {
    cudaMemPoolProps props;
    memset(&props, 0, sizeof(props));
    props.allocType = cudaMemAllocationTypePinned;
    props.handleTypes = cudaMemHandleTypeNone;
    props.location.type = cudaMemLocationTypeDevice;
    props.location.id = dev;
    cudaMemPool_t pool;
    e = cudaMemPoolCreate(&pool, &props);
    if (e != cudaSuccess) return e;
    unsigned long long thr = ~0ull;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    g_pool[dev] = pool;
  }
  *out = g_pool[dev];
  return cudaSuccess;
}
cudaError_t rt_ws_alloc(void** p, size_t bytes, cudaStream_t stream) {
  cudaMemPool_t pool;
  cudaError_t e = ws_pool(&pool);
  if (e != cudaSuccess) return e;
  return cudaMallocFromPoolAsync(p, bytes, pool, stream);
}
cudaError_t rt_ws_free(void* p, cudaStream_t stream) { return cudaFreeAsync(p, stream); }
static void ensure_pool_cached() {}

static int arg_error(const char* msg) {
  snprintf(g_err, sizeof(g_err), "argument error: %s", msg);
  return RT_ERR_ARG;
}
static int unsupported(const char* msg) {
  snprintf(g_err, sizeof(g_err), "unsupported: %s", msg);
  return RT_ERR_UNSUPPORTED;
}

// implemented in the kernel translation units
int rt_expm_batched_impl(const double*, const int32_t*, const double*, int, int, double*, cudaStream_t);
int rt_frechet_contract_impl(const double*, const int32_t*, const double*, const double*, int, int,
                             double*, cudaStream_t);
int rt_history_statistics_impl(const double*, const int32_t*, const double*, const double*, int, int, int,
                               double*, double*, double*, cudaStream_t);
int rt_expm_spectral_impl(const double*, const double*, const double*, const double*, const uint8_t*,
                          int, int, double*, cudaStream_t);
int rt_lb_transition_impl(const double*, const double*, int, int, double*, cudaStream_t);
int rt_support_sets_impl(int, int, int64_t, int64_t, int, const int32_t*, const double*, uint64_t*, cudaStream_t);
int rt_joint_distn_impl(int, int, int64_t, int64_t, const int32_t*, int, const double*, const void*,
                        const double*, const double*, const int8_t*, double*, double*, cudaStream_t);
int rt_prune_small_dispatch(int, int, bool, int64_t, int64_t, const int32_t*, int, int, int,
                            const double*, const double*, const void*, double*, int32_t*, double*,
                            int8_t*, double*, cudaStream_t);
int rt_prune_dmma_dispatch(int, int, bool, int64_t, int64_t, const int32_t*, int, int, int,
                           const double*, const double*, const void*, double*, int32_t*, double*,
                           int8_t*, double*, cudaStream_t);
int rt_posterior_small_dispatch(int, int, int64_t, int64_t, const int32_t*, int, int, int,
                                const int32_t*, const int32_t*, int,
                                const double*, const double*, const void*, const double*,
                                const int8_t*, double*, double*, double*, const double*, double*,
                                const double*, cudaStream_t);
int rt_posterior_dmma_dispatch(int, int, int64_t, int64_t, const int32_t*, const int32_t*, int,
                               const double*, const double*, const void*, const double*,
                               const int8_t*, double*, double*, double*, const double*, double*,
                               const double*, cudaStream_t);

int rt_raoteh_dispatch(const rt_raoteh_args&, cudaStream_t);

int rt_tmjp_dispatch(const rt_tmjp_args&, cudaStream_t);

int rt_posterior_draw_dispatch(const rt_posterior_draw_args&, cudaStream_t);
int rt_posterior_draw_mixture_dispatch(const rt_posterior_draw_mixture_args&, cudaStream_t);

extern "C" {

int rt_version(void) { return 205; }

int rt_release_workspace(void) {
  int dev = 0;
  RT_CUDA_CHECK(cudaGetDevice(&dev));
  if (dev >= 0 && dev < 64 && g_pool[dev]) {
    RT_CUDA_CHECK(cudaDeviceSynchronize());
    RT_CUDA_CHECK(cudaMemPoolTrimTo(g_pool[dev], 0));
  }
  return RT_OK;
}
const char* rt_last_error_string(void) { return g_err; }

int rt_expm_batched(const double* Q, const int32_t* q_index, const double* t, int n_mat, int S,
                    double* P, void* stream) {
  if (!Q || !t || !P) return arg_error("null pointer");
  if (S < 1 || S > 128) return unsupported("rt_expm_batched needs 1 <= S <= 128");
  ensure_pool_cached();
  return rt_expm_batched_impl(Q, q_index, t, n_mat, S, P, (cudaStream_t)stream);
}

int rt_frechet_contract(const double* Q, const int32_t* q_index, const double* t, const double* W,
                        int n_mat, int S, double* M, void* stream) {
  if (!Q || !t || !W || !M) return arg_error("null pointer");
  if (S < 1 || S > 64) return unsupported("rt_frechet_contract needs 1 <= S <= 64");
  ensure_pool_cached();
  return rt_frechet_contract_impl(Q, q_index, t, W, n_mat, S, M, (cudaStream_t)stream);
}

int rt_expm_spectral(const double* A, const double* lam, const double* B, const double* t,
                     const uint8_t* d_off, int n_mat, int S, double* P, void* stream) {
  if (!A || !lam || !B || !t || !P) return arg_error("null pointer");
  if (S < 1 || S > 64) return unsupported("rt_expm_spectral needs 1 <= S <= 64");
  return rt_expm_spectral_impl(A, lam, B, t, d_off, n_mat, S, P, (cudaStream_t)stream);
}

int rt_lb_transition(const double* Q, const double* t, int n_mat, int S, double* P, void* stream) {
  if (!Q || !t || !P) return arg_error("null pointer");
  if (S < 1 || S > 1024) return unsupported("rt_lb_transition needs 1 <= S <= 1024");
  return rt_lb_transition_impl(Q, t, n_mat, S, P, (cudaStream_t)stream);
}

int rt_history_statistics(const double* Q, const int32_t* q_index, const double* t, const double* W,
                          int n_mat, int first, int S, double* M, double* dwell, double* trans,
                          void* stream) {
  if (!Q || !t || !W || !M || !dwell || !trans) return arg_error("null pointer");
  if (S < 1 || S > 64) return unsupported("rt_history_statistics needs 1 <= S <= 64");
  if (first < 0 || first > n_mat) return arg_error("first out of range");
  ensure_pool_cached();
  return rt_history_statistics_impl(Q, q_index, t, W, n_mat, first, S, M, dwell, trans,
                                    (cudaStream_t)stream);
}

int rt_support_sets(int S, int n_nodes, int64_t n_sites, int64_t site_stride, int passes,
                    const int32_t* parent, const double* P, uint64_t* mask, void* stream) {
  if (!parent || !P || !mask) return arg_error("null pointer");
  if (site_stride < n_sites) return arg_error("site_stride < n_sites");
  if (passes < 1 || passes > 3) return arg_error("passes must be 1 (backward), 2 (forward) or 3");
  ensure_pool_cached();
  return rt_support_sets_impl(S, n_nodes, n_sites, site_stride, passes, parent, P, mask,
                              (cudaStream_t)stream);
}

int rt_joint_distn(int S, int n_nodes, int64_t n_sites, int64_t site_stride, const int32_t* edges,
                   int n_edges, const double* P, int obs_kind, const void* obs,
                   const double* partials, const double* node_distn, const int8_t* status,
                   double* J, double* D_all, void* stream) {
  if (!edges || !P || !partials || !node_distn || !status || !J || !D_all)
    return arg_error("null pointer");
  if (obs_kind < 0 || obs_kind > 2) return arg_error("obs_kind");
  (void)n_nodes;
  return rt_joint_distn_impl(S, obs_kind, n_sites, site_stride, edges, n_edges, P, obs, partials,
                             node_distn, status, J, D_all, (cudaStream_t)stream);
}

int rt_prune_loglik(int S, int n_nodes, int64_t n_sites, int64_t site_stride,
                    const int32_t* program, int n_ops, int n_slots, const double* P,
                    const double* root_distn, int obs_kind, const void* obs, double* partials,
                    int32_t* exponents, double* loglik, int8_t* status, double* loglik_sum,
                    void* stream) {
  if (!program || !P || !loglik || !status) return arg_error("null pointer");
  if (obs_kind < 0 || obs_kind > 3) return arg_error("obs_kind");
  if (obs_kind == 3 && !(S >= 2 && S <= 8)) return unsupported("RT_OBS_CODES4 needs 2 <= S <= 8");
  if (site_stride < n_sites) return arg_error("site_stride < n_sites");
  if (n_sites <= 0) return RT_OK;
  if (n_ops <= 0 || n_slots <= 0 || n_nodes <= 1) return arg_error("empty program");
  const bool store = partials != nullptr;
  ensure_pool_cached();
  int rc;
  if (S >= 2 && S <= 8)
    rc = rt_prune_small_dispatch(S, obs_kind, store, n_sites, site_stride, program, n_ops, n_slots,
                                 n_nodes, P, root_distn, obs, partials, exponents, loglik, status,
                                 loglik_sum, (cudaStream_t)stream);
  else if (S >= 1 && S <= 64)
    rc = rt_prune_dmma_dispatch(S, obs_kind, store, n_sites, site_stride, program, n_ops, n_slots,
                                n_nodes, P, root_distn, obs, partials, exponents, loglik, status,
                                loglik_sum, (cudaStream_t)stream);
  else
    return unsupported("rt_prune_loglik needs 1 <= S <= 64");
  if (rc == RT_ERR_UNSUPPORTED) snprintf(g_err, sizeof(g_err), "unsupported: shared-memory budget exceeded");
  return rc;
}

static int posterior_common(int S, int n_nodes, int64_t n_sites, int64_t site_stride,
                            const int32_t* program, int n_ops, int n_slots,
                            const int32_t* edges, const int32_t* level_ptr_h, int n_levels,
                            const double* P, const double* root_distn, int obs_kind, const void* obs,
                            const double* partials, const int8_t* status, double* node_distn, double* W,
                            double* root_post_sum, const double* K, double* branch_out,
                            const double* site_weight, void* stream) {
  if (!edges || !level_ptr_h || !P || !partials || !status || !W)
    return arg_error("null pointer");
  if (!node_distn && !(S >= 2 && S <= 8 && program))
    return arg_error("node_distn may be NULL only for S <= 8 with the upward program given");
  if (obs_kind < 0 || obs_kind > 3) return arg_error("obs_kind");
  if (obs_kind == 3 && !(S >= 2 && S <= 8 && program)) return unsupported("RT_OBS_CODES4 needs 2 <= S <= 8");
  if (site_stride < n_sites) return arg_error("site_stride < n_sites");
  if ((K == nullptr) != (branch_out == nullptr)) return arg_error("K and branch_out go together");
  if (site_weight && branch_out) return arg_error("site weights with per-branch output");
  if (n_sites <= 0) return RT_OK;
  int rc;
  if (S >= 2 && S <= 8)
    rc = rt_posterior_small_dispatch(S, obs_kind, n_sites, site_stride, program, n_ops, n_slots,
                                     n_nodes, edges, level_ptr_h, n_levels, P, root_distn, obs,
                                     partials, status, node_distn, W, root_post_sum, K, branch_out,
                                     site_weight, (cudaStream_t)stream);
  else if (S >= 1 && S <= 64)
    rc = rt_posterior_dmma_dispatch(S, obs_kind, n_sites, site_stride, edges, level_ptr_h,
                                    n_levels, P, root_distn, obs, partials, status, node_distn, W,
                                    root_post_sum, K, branch_out, site_weight, (cudaStream_t)stream);
  else
    return unsupported("rt_posterior_stats needs 1 <= S <= 64");
  if (rc == RT_ERR_UNSUPPORTED) snprintf(g_err, sizeof(g_err), "unsupported: shared-memory budget");
  return rc;
}

int rt_posterior_stats(int S, int n_nodes, int64_t n_sites, int64_t site_stride,
                       const int32_t* program, int n_ops, int n_slots,
                       const int32_t* edges, const int32_t* level_ptr_h, int n_levels,
                       const double* P, const double* root_distn, int obs_kind, const void* obs,
                       const double* partials, const int8_t* status, double* node_distn, double* W,
                       double* root_post_sum, void* stream) {
  return posterior_common(S, n_nodes, n_sites, site_stride, program, n_ops, n_slots, edges,
                          level_ptr_h, n_levels, P, root_distn, obs_kind, obs, partials, status,
                          node_distn, W, root_post_sum, nullptr, nullptr, nullptr, stream);
}

int rt_posterior_weighted_stats(int S, int n_nodes, int64_t n_sites, int64_t site_stride,
                                const int32_t* program, int n_ops, int n_slots,
                                const int32_t* edges, const int32_t* level_ptr_h, int n_levels,
                                const double* P, const double* root_distn, int obs_kind,
                                const void* obs, const double* partials, const int8_t* status,
                                double* node_distn, double* W, double* root_post_sum,
                                const double* site_weight, void* stream) {
  if (!site_weight) return arg_error("null pointer");
  return posterior_common(S, n_nodes, n_sites, site_stride, program, n_ops, n_slots, edges,
                          level_ptr_h, n_levels, P, root_distn, obs_kind, obs, partials, status,
                          node_distn, W, root_post_sum, nullptr, nullptr, site_weight, stream);
}

int rt_posterior_branch_stats(int S, int n_nodes, int64_t n_sites, int64_t site_stride,
                              const int32_t* program, int n_ops, int n_slots,
                              const int32_t* edges, const int32_t* level_ptr_h, int n_levels,
                              const double* P, const double* root_distn, int obs_kind,
                              const void* obs, const double* partials, const int8_t* status,
                              double* node_distn, double* W, double* root_post_sum,
                              const double* K, double* branch_out, void* stream) {
  if (!K || !branch_out) return arg_error("null pointer");
  return posterior_common(S, n_nodes, n_sites, site_stride, program, n_ops, n_slots, edges,
                          level_ptr_h, n_levels, P, root_distn, obs_kind, obs, partials, status,
                          node_distn, W, root_post_sum, K, branch_out, nullptr, stream);
}

int rt_copy2d_async(void* dst, size_t dst_pitch, const void* src, size_t src_pitch,
                    size_t width_bytes, size_t height, int to_device, void* stream) {
  if (!dst || !src) return arg_error("null pointer");
  RT_CUDA_CHECK(cudaMemcpy2DAsync(dst, dst_pitch, src, src_pitch, width_bytes, height,
                                  to_device ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost,
                                  (cudaStream_t)stream));
  return RT_OK;
}

}  // extern "C"

static int raoteh_run_impl(const rt_raoteh_args& R, void* stream) {
  if (!R.program || !R.parent || !R.length || !R.B || !R.rate || !R.obs || !R.node_state ||
      !R.ev_time || !R.ev_sb || !R.ev_count || !R.ev_total || !R.status)
    return arg_error("null pointer");
  if (R.obs_kind != 0 && R.obs_kind != 1) return arg_error("rt_raoteh_sweeps takes codes or masks");
  if (R.traj_stride < R.n_traj || R.n_sites <= 0 || R.cap <= 0) return arg_error("sizes");
  if (R.n_traj <= 0) return RT_OK;
  const int S = R.S;
  if (S == 7 || (S >= 9 && S <= 64)) {
    if (R.time_f64) return unsupported("fp64 event times: S in {2,3,4,5,6,8} only");
    if (R.sweep_count) return unsupported("sweep_count: S in {2,3,4,5,6,8} only");
    // warp-per-trajectory kernel (csrc/rt_tmjp.cu) on the same trajectory layout
    rt_tmjp_args A;
    memset(&A, 0, sizeof(A));
    A.S = S; A.n_parts = 0; A.n_nodes = R.n_nodes; A.n_ops = R.n_ops; A.n_slots = R.n_slots;
    A.cap_p = R.cap; A.cap_t = 1; A.obs_kind = R.obs_kind;
    A.program = R.program; A.parent = R.parent; A.length = R.length; A.B = R.B; A.rate_p = R.rate;
    A.pi_p = R.root_distn; A.obs = R.obs; A.obs_stride = R.obs_stride;
    A.n_traj = R.n_traj; A.n_sites = R.n_sites; A.traj0 = R.traj0;
    A.p_node = R.node_state; A.p_cnt = R.ev_count; A.pn_traj_stride = 1; A.pn_node_stride = R.traj_stride;
    A.p_total = R.ev_total; A.p_time = (float*)R.ev_time; A.p_sb = R.ev_sb; A.status = R.status;
    A.seed = R.seed; A.sweep0 = R.sweep0; A.n_sweeps = R.n_sweeps;
    A.mode = R.init_k >= 0 ? RT_TMJP_INIT_PRIMARY : RT_TMJP_SWEEP; A.init_k = R.init_k;
    const bool st = R.dwell_sum != nullptr && R.trans_sum != nullptr && R.init_k < 0;
    A.flags = st ? RT_TMJP_F_STATS_PRIMARY : 0;
    A.prim_dwell = R.dwell_sum; A.prim_trans = R.trans_sum;
    int rc = rt_tmjp_dispatch(A, (cudaStream_t)stream);
    if (rc == RT_ERR_UNSUPPORTED) snprintf(g_err, sizeof(g_err), "unsupported: shared-memory budget");
    return rc;
  }
  int rc = rt_raoteh_dispatch(R, (cudaStream_t)stream);
  if (rc == RT_ERR_UNSUPPORTED) snprintf(g_err, sizeof(g_err), "unsupported: S or shared-memory budget");
  return rc;
}

extern "C" {

int rt_raoteh_run(const rt_raoteh_args* args, void* stream) {
  if (!args) return arg_error("null pointer");
  return raoteh_run_impl(*args, stream);
}

int rt_raoteh_sweeps(int S, int n_nodes, int64_t n_traj, int64_t traj_stride, int64_t n_sites,
                     int64_t traj0, const int32_t* program, int n_ops, int n_slots,
                     const int32_t* parent, const double* length, const double* B,
                     const double* rate, const double* root_distn, int obs_kind, const void* obs,
                     int64_t obs_stride, uint8_t* node_state, float* ev_time, uint8_t* ev_sb,
                     uint8_t* ev_count, int32_t* ev_total, int cap, uint64_t seed, int64_t sweep0,
                     int n_sweeps, int init_k, double* dwell_sum, double* trans_sum, int8_t* status,
                     void* stream) {
  rt_raoteh_args R;
  memset(&R, 0, sizeof(R));
  R.S = S; R.n_nodes = n_nodes; R.n_ops = n_ops; R.n_slots = n_slots; R.obs_kind = obs_kind;
  R.cap = cap; R.n_sweeps = n_sweeps; R.init_k = init_k;
  R.n_traj = n_traj; R.traj_stride = traj_stride; R.n_sites = n_sites; R.traj0 = traj0;
  R.obs_stride = obs_stride; R.sweep0 = sweep0; R.seed = seed;
  R.program = program; R.parent = parent; R.length = length; R.B = B; R.rate = rate;
  R.root_distn = root_distn; R.obs = obs; R.node_state = node_state; R.ev_time = ev_time;
  R.ev_sb = ev_sb; R.ev_count = ev_count; R.ev_total = ev_total;
  R.dwell_sum = dwell_sum; R.trans_sum = trans_sum; R.status = status;
  return raoteh_run_impl(R, stream);
}

}  // extern "C"

// the checks of rt_posterior_draw; RT_OK if the arguments are valid
static int posterior_draw_check(const rt_posterior_draw_args& R) {
  if (!R.program || !R.parent || !R.length || !R.Q || !R.P || !R.obs || !R.partials ||
      !R.node_state || !R.ev_time || !R.ev_sb || !R.ev_count || !R.ev_total || !R.status)
    return arg_error("null pointer");
  if ((R.dwell_sum == nullptr) != (R.trans_sum == nullptr)) return arg_error("dwell_sum and trans_sum go together");
  if (R.obs_kind != 0 && R.obs_kind != 1) return arg_error("rt_posterior_draw takes codes or masks");
  if (R.S < 2 || R.S > 8) return unsupported("rt_posterior_draw needs 2 <= S <= 8");
  if (R.time_f64 && R.S == 7) return unsupported("fp64 event times: S in {2,3,4,5,6,8} only");
  if (R.traj_stride < R.n_traj || R.n_sites <= 0 || R.cap <= 0) return arg_error("sizes");
  if (R.site_stride < R.n_sites) return arg_error("site_stride < n_sites");
  if (R.k < 0 || R.k >= INT32_MAX) return arg_error("draw index k out of range");
  if (R.n_ops <= 0 || R.n_nodes <= 1) return arg_error("empty program");
  return RT_OK;
}

extern "C" {

int rt_posterior_draw(const rt_posterior_draw_args* args, void* stream) {
  if (!args) return arg_error("null pointer");
  const rt_posterior_draw_args& R = *args;
  int rc = posterior_draw_check(R);
  if (rc != RT_OK) return rc;
  if (R.n_traj <= 0) return RT_OK;
  rc = rt_posterior_draw_dispatch(R, (cudaStream_t)stream);
  if (rc == RT_ERR_UNSUPPORTED) snprintf(g_err, sizeof(g_err), "unsupported: S or shared-memory budget");
  return rc;
}

int rt_posterior_draw_mixture(const rt_posterior_draw_mixture_args* args, void* stream) {
  if (!args) return arg_error("null pointer");
  const rt_posterior_draw_mixture_args& M = *args;
  int rc = posterior_draw_check(M.base);
  if (rc != RT_OK) return rc;
  if (M.K < 1 || M.K > 255) return arg_error("rt_posterior_draw_mixture needs 1 <= K <= 255");
  if (!M.class_post || !M.site_class) return arg_error("null pointer");
  if (M.class_post_stride < M.base.n_sites) return arg_error("class_post_stride < n_sites");
  if (M.partials_class_stride < 0) return arg_error("partials_class_stride < 0");
  if (M.base.sweep_count) return arg_error("rt_posterior_draw_mixture takes no sweep_count");
  if (M.base.n_traj <= 0) return RT_OK;
  rc = rt_posterior_draw_mixture_dispatch(M, (cudaStream_t)stream);
  if (rc == RT_ERR_UNSUPPORTED) snprintf(g_err, sizeof(g_err), "unsupported: S or shared-memory budget");
  return rc;
}

}  // extern "C"

int rt_forward_simulate_dispatch(const rt_forward_args&, cudaStream_t);

extern "C" {

int rt_forward_simulate(const rt_forward_args* args, void* stream) {
  if (!args) return arg_error("null pointer");
  const rt_forward_args& R = *args;
  if (R.S < 2 || R.S > 64) return unsupported("rt_forward_simulate needs 2 <= S <= 64");
  if (R.K < 1 || R.K > 255) return arg_error("rt_forward_simulate needs 1 <= K <= 255");
  if (R.mode != RT_SIM_NODES && R.mode != RT_SIM_HISTORY) return arg_error("mode");
  if (!R.program || !R.parent) return arg_error("null pointer");
  if (R.K > 1 && !R.class_weight) return arg_error("class_weight is required when K > 1");
  if (R.obs && !R.obs_slot) return arg_error("obs needs obs_slot");
  if (R.tmpl && !R.obs) return arg_error("tmpl without obs");
  if (R.n_ops <= 0 || R.n_nodes <= 1) return arg_error("empty program");
  if (R.n_traj < 0 || R.traj0 < 0 || R.traj_stride < R.n_traj) return arg_error("traj_stride < n_traj");
  if (R.obs && R.obs_stride < R.n_traj) return arg_error("obs_stride < n_traj");
  if (R.tmpl && (R.tmpl_n_sites <= 0 || R.tmpl_stride < R.tmpl_n_sites)) return arg_error("tmpl_stride / tmpl_n_sites");
  if (R.k < 0 || R.k >= INT32_MAX) return arg_error("replicate index k out of range");
  if (R.mode == RT_SIM_NODES) {
    if (!R.P) return arg_error("null pointer");
  } else {
    if (!R.Q || !R.length || !R.node_state || !R.ev_time || !R.ev_sb || !R.ev_count || !R.ev_total ||
        !R.status)
      return arg_error("null pointer");
    if ((R.dwell_sum == nullptr) != (R.trans_sum == nullptr)) return arg_error("dwell_sum and trans_sum go together");
    if (R.cap <= 0) return arg_error("cap");
    if (R.time_f64 && (R.S == 7 || R.S > 8)) return unsupported("fp64 event times: S in {2,3,4,5,6,8} only");
  }
  if (R.n_traj == 0) return RT_OK;
  int rc = rt_forward_simulate_dispatch(R, (cudaStream_t)stream);
  if (rc == RT_ERR_UNSUPPORTED)
    snprintf(g_err, sizeof(g_err), "unsupported: shared-memory budget (tree size, or K S (8 + 4 S) bytes of statistics)");
  return rc;
}

}  // extern "C"

extern "C" {

int rt_tmjp_run(const rt_tmjp_args* a, void* stream) {
  if (!a) return arg_error("null pointer");
  const rt_tmjp_args& A = *a;
  if (!A.program || !A.parent || !A.length || !A.B || !A.rate_p || !A.obs || !A.p_node ||
      !A.p_cnt || !A.p_total || !A.p_time || !A.p_sb || !A.status)
    return arg_error("null pointer");
  if (A.S < 2 || A.S > 64) return unsupported("rt_tmjp_run needs 2 <= S <= 64");
  if (A.n_parts < 0 || A.n_parts > 32) return unsupported("rt_tmjp_run needs n_parts <= 32");
  if (A.n_parts > 0 && (!A.part || !A.absorb || !A.t_node || !A.t_cnt || !A.t_total || !A.t_time))
    return arg_error("tolerance arrays missing");
  if (A.n_parts > 0 && (!(A.rate_on > 0) || !(A.rate_off >= 0) || !(A.omega_t > 0)))
    return arg_error("tolerance rates");
  if (A.tol_obs && !A.tol_obs_slot) return arg_error("tol_obs without tol_obs_slot");
  if (A.obs_kind != 0 && A.obs_kind != 1) return arg_error("rt_tmjp_run takes codes or masks");
  if (A.cap_p <= 0 || A.cap_p > 4096 || A.cap_t <= 0 || A.cap_t > 255) return arg_error("capacities");
  if ((int64_t)(A.n_parts + 2) * (A.n_ops + 1) >= 65536) return unsupported("program too long");
  if (A.mode < 0 || A.mode > 4) return arg_error("mode");
  if (A.mode == RT_TMJP_TRAJ_LOGLIK && (!A.traj_loglik || !(A.omega_p > 0))) return arg_error("traj_loglik / omega_p");
  if ((A.mode == RT_TMJP_INIT_TOLERANCE || A.mode == RT_TMJP_SUMMARY) && A.n_parts == 0)
    return arg_error("mode needs tolerance classes");
  if (A.n_traj <= 0) return RT_OK;
  ensure_pool_cached();
  int rc = rt_tmjp_dispatch(A, (cudaStream_t)stream);
  if (rc == RT_ERR_UNSUPPORTED) snprintf(g_err, sizeof(g_err), "unsupported: shared-memory budget");
  return rc;
}

}  // extern "C"
