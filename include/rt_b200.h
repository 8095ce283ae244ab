/*
 * rt_b200.h -- C ABI of librt_b200.so: the B200-native replacement for the
 * native calls on raoteh's data-parallel hot path.
 *
 * The reference's only native boundary is Python -> `pyfelscore` (Cython,
 * un-vendored; README.md:8-9).  Each entry point below is the BATCHED
 * (many sites / chains per call) replacement of one or more of those calls
 * and of the scipy calls around them; the reference interface replaced is
 * cited per function (paths relative to the reference root).
 *
 * Conventions
 *   - plain C types only; every array argument is a DEVICE pointer into
 *     caller-owned memory unless its name ends in `_h` (host pointer);
 *   - `stream` is a cudaStream_t passed as void*; calls are asynchronous on
 *     it, hold no global state and are re-entrant per stream;
 *   - return value: RT_OK (0) or an RT_ERR_* code; rt_last_error_string()
 *     describes the last failure on the calling thread;
 *   - nodes are numbered in DFS preorder from the root (root = 0,
 *     parent < child), per-edge matrices are indexed by the CHILD node
 *     (slot 0 unused) -- the reference's own convention for its native calls
 *     (raoteh/sampler/_density.py:104-180);
 *   - site-major arrays are laid out [row][site] with `site_stride` elements
 *     between rows (site-minor => coalesced), states 0..S-1;
 *   - per-site status (int8): 0 ok, 1 structural zero, 2 numerical zero
 *     (raoteh/sampler/_util.py:14-21: StructuralZeroProb / NumericalZeroProb).
 */
#ifndef RT_B200_H
#define RT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RT_OK 0
#define RT_ERR_ARG 1
#define RT_ERR_CUDA 2
#define RT_ERR_UNSUPPORTED 3

/* observation encodings (argument `obs_kind`) */
#define RT_OBS_CODES 0 /* uint8  [n_obs][site_stride]     hard state, 255 = unobserved */
#define RT_OBS_MASK 1  /* uint64 [n_obs][site_stride]     bitmask of allowed states     */
#define RT_OBS_DENSE 2 /* double [n_obs][S][site_stride]  emission likelihoods          */
#define RT_OBS_CODES4 3 /* uint8 [n_obs][(site_stride+1)/2] two hard states per byte (site i in
                           nibble i & 1 of byte i >> 1), 15 = unobserved; S <= 8, rt_prune_loglik and
                           rt_posterior_stats only: halves the host-to-device bytes of nucleotide data */

int rt_version(void);
const char* rt_last_error_string(void);

/*
 * Per-call workspaces (expm scratch, Rao-Teh event records, ...) come from a PRIVATE
 * stream-ordered memory pool per device, created on first use; the device's default pool and
 * its attributes are never touched.  Freed workspaces stay cached in that pool between calls.
 * rt_release_workspace() synchronises the device and returns the cached memory to the driver.
 * Largest workspace: rt_raoteh_sweeps, min(n_traj, 2^19) x cap x (8 S + 16) bytes (trajectories
 * are processed in launches of 2^19); rt_tmjp_run sizes its scratch by resident warps.
 */
int rt_release_workspace(void);

/*
 * P[m] = expm(Q[q_index[m]] * t[m]),  m = 0..n_mat-1   (S <= 128)
 * Q: [n_q][S][S] row-major with diagonal; q_index: [n_mat] or NULL (all use Q[0]).
 * Replaces scipy.linalg.expm called once per edge PER SITE at
 * raoteh/sampler/_mjp_dense.py:357 (custom_expm :24) and _linalg.py:81
 * (sparse_expm_naive), and pyfelscore.get_tolerance_rate_matrix
 * (_tmjp_dense.py:239) / get_mmpp_block (_linalg.py:44-46) for S = 3.
 */
int rt_expm_batched(const double* Q, const int32_t* q_index, const double* t,
                    int n_mat, int S, double* P, void* stream);

/*
 * P[m] = A diag(exp(t[m] * lam)) B for m in [0, n_mat): transition matrices of a time-reversible
 * rate matrix from its spectral decomposition (A, lam, B double [S][S], [S], [S][S]; S <= 64),
 * d_off (nullable, uint8 [S]): states whose diagonal entry is forced to 1.
 * Replaces getp_spectral_v2 / reconstruct_spectral_v2 called once per branch
 * (examples/p53/qtop.py:76-85, 283-288; decomposition qtop.py:126-148 stays on the host).
 */
int rt_expm_spectral(const double* A, const double* lam, const double* B, const double* t,
                     const uint8_t* d_off, int n_mat, int S, double* P, void* stream);

/*
 * P[m] = small-step LOWER BOUND of expm(Q t[m]), m in [0, n_mat): the probability of no change on
 * the diagonal and of exactly one change a -> b off it (Q: [S][S] with diagonal).
 * Replaces pyfelscore.get_lb_transition_matrix (examples/p53/liwen.py:43-46; spec getp_lb :48-82).
 */
int rt_lb_transition(const double* Q, const double* t, int n_mat, int S, double* P, void* stream);

/*
 * M[m] = L(t[m] Q^T, t[m] W[m]) -- Frechet derivative of expm; equals
 * sum_ab W[m][a][b] * expm_frechet(tQ, t E_cd)[a][b] at entry [c][d].  (S <= 64)
 * Replaces the S + nnz(Q) scipy.linalg.expm_frechet calls per edge per site at
 * raoteh/sampler/_mjp_dense.py:497-520 (sparse twin _mjp.py:531-580) and
 * pyfelscore.get_mmpp_frechet_* (_linalg.py:107-118) /
 * get_tolerance_expectations (_tmjp_dense.py:339).
 */
int rt_frechet_contract(const double* Q, const int32_t* q_index, const double* t,
                        const double* W, int n_mat, int S, double* M, void* stream);

/*
 * rt_frechet_contract followed by the accumulation over edges, in one call:
 *   M[m] as above for m in [0, n_mat), M[m] = 0 for m < first (the root slot has no edge);
 *   dwell[c]    = sum_{m >= first} M[m][c][c]                         (double [S])
 *   trans[c][d] = sum_{m >= first} Q[q_index[m]][c][d] * M[m][c][d]   (c != d; 0 on the diagonal; [S][S])
 * Replaces the loop over edges of _mjp_dense.get_expected_history_statistics
 * (raoteh/sampler/_mjp_dense.py:497-533: dwell times :521-526, transition counts :527-533).
 */
int rt_history_statistics(const double* Q, const int32_t* q_index, const double* t,
                          const double* W, int n_mat, int first, int S, double* M,
                          double* dwell, double* trans, void* stream);

/*
 * Structural support of every node for every site (integer work):
 * backward pass (state kept iff every child has a reachable kept state) then
 * forward pass (state kept iff reachable from a kept parent state).
 * passes: 1 = backward only (the reference's "pset"), 3 = backward then forward ("set").
 * mask: uint64 [n_nodes][site_stride] in/out; parent: int32 [n_nodes];
 * P: [n_nodes][S][S] (only the > 0 pattern is used).  S <= 64.
 * Replaces pyfelscore.mcy_esd_get_node_to_pset + esd_get_node_to_set
 * (raoteh/sampler/_mcy_dense.py:168-179,270-281; _mcy.py:219-230,508-519;
 * specs _mcy.py:397-470 and _mc0.py:89-138) and the shared-pattern variants
 * mcy_get_node_to_pset / get_node_to_set (_mcy.py:158-174).
 */
int rt_support_sets(int S, int n_nodes, int64_t n_sites, int64_t site_stride, int passes,
                    const int32_t* parent, const double* P, uint64_t* mask, void* stream);

/*
 * Felsenstein pruning + root combine, batched over sites.
 *   L[a,s] = obs[a,s] * prod_{b in ch(a)} sum_s' P_b[s,s'] L[b,s'];
 *   loglik = log(sum_s pi[s] L[root,s])      (pi = 1 if root_distn == NULL)
 * program: int32 [n_ops][4] upward program (see raoteh_b200/lowering.py),
 * n_slots its stack depth.  partials (nullable): [n_store][S][site_stride]
 * scaled partials of the internal nodes, exponents (nullable):
 * [n_store][site_stride] with true partial = partial * 2^exponent.
 * loglik: [n_sites]; status: [n_sites]; loglik_sum (nullable): [1], += sum of
 * the finite log-likelihoods (the value the site-sharded job allreduces).
 * Replaces pyfelscore.mcy_esd_get_node_to_pmap (raoteh/sampler/_mcy_dense.py:
 * 184-189,286-291; _mcy.py:533-538; spec _mcy.py:611-682; emission form
 * _mcz.py:94-166) + _mc0_dense.get_likelihood (_mc0_dense.py:147-212).
 */
int rt_prune_loglik(int S, int n_nodes, int64_t n_sites, int64_t site_stride,
                    const int32_t* program, int n_ops, int n_slots,
                    const double* P, const double* root_distn,
                    int obs_kind, const void* obs,
                    double* partials, int32_t* exponents,
                    double* loglik, int8_t* status, double* loglik_sum, void* stream);

/*
 * Downward pass + sufficient statistics, batched over sites.
 *   D[root] = norm(pi * L_root); for each edge (a -> b):
 *   G_b = D[a] / (P_b L_b);  D[b] = L_b * (P_b^T G_b);
 *   W[b] += sum_sites G_b (x) L_b   restricted to P_b > 0   (= sum J_b / P_b)
 * edges: int32 [n_edges][4] downward program rows (child node, parent store
 * idx, child store idx or -1, child obs slot), sorted by depth of the child;
 * level_ptr_h: HOST int32 [n_levels+1], rows level_ptr_h[l]..level_ptr_h[l+1]
 * form level l (one launch per level: parents before children).
 * program / n_ops / n_slots: the upward program (as for rt_prune_loglik); for
 * S <= 8 the kernel walks it backwards per site (no level launches, marginals
 * stay on chip) and node_distn may then be NULL when only statistics are wanted.
 * partials: from rt_prune_loglik; node_distn: [n_store][S][site_stride] out
 * (posterior marginals of the internal nodes); W: [n_nodes][S][S], += ;
 * root_post_sum (nullable): [S], += sum_sites D[root].
 * Sites whose status != 0 are skipped.
 * Replaces pyfelscore.mc0_esd_get_node_to_distn (raoteh/sampler/
 * _mc0_dense.py:381, _mcy_dense.py:195; spec _mc0_dense.py:400-489) and
 * mc0_esd_get_joint_endpoint_distn (_mcy_dense.py:205; spec
 * _mc0_dense.py:217-270); the joint J is consumed on chip (never stored).
 */
int rt_posterior_stats(int S, int n_nodes, int64_t n_sites, int64_t site_stride,
                       const int32_t* program, int n_ops, int n_slots,
                       const int32_t* edges, const int32_t* level_ptr_h, int n_levels,
                       const double* P, const double* root_distn,
                       int obs_kind, const void* obs,
                       const double* partials, const int8_t* status,
                       double* node_distn, double* W, double* root_post_sum, void* stream);

/*
 * rt_posterior_stats with one weight per site: the root marginal becomes
 *   D[root] = w_site * norm(pi * L_root),
 * and since nothing below the root renormalises, W, root_post_sum and node_distn all carry the
 * weight (each site contributes w_site times what rt_posterior_stats adds).  A site with weight 0
 * contributes nothing.  site_weight: device fp64, required, entries [0, n_sites) read (indexed
 * like status); weights are meant to be non-negative and finite.  Uses: the E-step of site-class mixtures (w = posterior probability
 * of the class at the site) and site-pattern compression (w = number of alignment columns with
 * the pattern).
 */
int rt_posterior_weighted_stats(int S, int n_nodes, int64_t n_sites, int64_t site_stride,
                                const int32_t* program, int n_ops, int n_slots,
                                const int32_t* edges, const int32_t* level_ptr_h, int n_levels,
                                const double* P, const double* root_distn,
                                int obs_kind, const void* obs,
                                const double* partials, const int8_t* status,
                                double* node_distn, double* W, double* root_post_sum,
                                const double* site_weight, void* stream);

/*
 * rt_posterior_stats plus, per SITE and BRANCH, the posterior expectation of a statistic
 * given by one S x S kernel per edge:
 *   branch_out[b][site] = sum_ac J_b[a,c] K_b[a,c] / P_b[a,c] = sum_ac G_b[a] K_b[a,c] L_b[c]
 * K: [n_nodes][S][S] (slot 0 unused), branch_out: [n_nodes][site_stride] (row 0 not written).
 * With K_b = L(t_b Q, t_b (E o Q)) (one rt_frechet_contract call) this is the expected number
 * of E-type transitions on every branch for every site -- the per-branch tables of
 * examples/code2x3/extras.py:19-132 (get_expected_ntransitions) and
 * examples/p53/liwen-branch-expectation.py:176-356 (synonymous / non-synonymous counts per
 * branch and codon column), which the reference computes one site and one branch at a time.
 */
int rt_posterior_branch_stats(int S, int n_nodes, int64_t n_sites, int64_t site_stride,
                              const int32_t* program, int n_ops, int n_slots,
                              const int32_t* edges, const int32_t* level_ptr_h, int n_levels,
                              const double* P, const double* root_distn,
                              int obs_kind, const void* obs,
                              const double* partials, const int8_t* status,
                              double* node_distn, double* W, double* root_post_sum,
                              const double* K, double* branch_out, void* stream);

/*
 * Pitched host<->device copy on `stream` (cudaMemcpy2DAsync): moves a chunk of sites
 * [row][lo:hi] of a site-minor array between a pinned HOST array and the device
 * array without staging, so chunk k+1 can be copied under the kernels of chunk k.
 * to_device != 0: `src` is the host pointer; else `dst` is.
 */
int rt_copy2d_async(void* dst, size_t dst_pitch, const void* src, size_t src_pitch,
                    size_t width_bytes, size_t height, int to_device, void* stream);

/*
 * Materialised per-edge joints and all-node marginals for small batches
 * (n_sites <= 65535):  J[b][site][a][c] = D[parent(b)][a] * norm(P_b[a,:] L_b)[c],
 * D_all[b][site][c] = sum_a J[b][site][a][c].  edges: all rows of the downward
 * program; partials / node_distn as produced by rt_prune_loglik /
 * rt_posterior_stats.  J: [n_nodes][n_sites][S][S], D_all: [n_nodes][n_sites][S]
 * (rows of the root are not written).
 * Replaces pyfelscore.mc0_esd_get_joint_endpoint_distn (raoteh/sampler/
 * _mcy_dense.py:205; spec _mc0_dense.py:217-270) where the caller wants J itself
 * (_mc0_dense.get_joint_endpoint_distn, _mcy_dense.kitchen_sink :57).
 */
int rt_joint_distn(int S, int n_nodes, int64_t n_sites, int64_t site_stride,
                   const int32_t* edges, int n_edges, const double* P,
                   int obs_kind, const void* obs, const double* partials,
                   const double* node_distn, const int8_t* status,
                   double* J, double* D_all, void* stream);

/*
 * Rao-Teh uniformization sweeps for n_traj independent trajectories
 * (trajectory t = chain * n_sites + site; observations are per site:
 * site = (traj0 + t) % n_sites), n_sweeps sweeps per call, Philox4x32-10
 * keyed by (seed; traj0 + t, sweep0 + i) so results do not depend on how
 * trajectories are split over launches or GPUs.  2 <= S <= 64: S in {2,3,4,5,6,8}
 * runs one thread per trajectory; S = 7 and 9 <= S <= 64 run the warp-per-trajectory
 * kernel below, which has neither option of rt_raoteh_run (time_f64, sweep_count).
 *
 * Trajectory state (caller-owned device arrays, trajectory-minor):
 *   node_state uint8 [n_nodes][traj_stride]  state at every tree node
 *   ev_count   uint8 [n_nodes][traj_stride]  real jumps on the edge above node b
 *   ev_total   int32 [traj_stride]           total real jumps
 *   ev_time    float [traj_stride][cap]      jump times from the PARENT end of the
 *   ev_sb      uint8 [traj_stride][cap]      edge / state on the parent side; the
 *              jumps of a trajectory are contiguous and occupy entries
 *              [cap - ev_total, cap) in upward-program order (edges in program
 *              order, child end first).
 * B = I + Q/omega, rate[s] = omega - q_s (raoteh/sampler/_sampler.py:346-355).
 * init_k >= 0: build an initial history with init_k equally spaced events on
 * every edge (one round of _sampler.get_restricted_feasible_history,
 * raoteh/sampler/_sampler.py:612-643); status 1 where infeasible.
 * init_k < 0: n_sweeps Rao-Teh sweeps (raoteh/sampler/_sampler.py:366-390 =
 * _sample_mjp.resample_poisson :19 + _sample_mcy.resample_edge_states :86 +
 * _graph_transform.remove_redundant_nodes :144); dwell_sum[S] / trans_sum[S*S]
 * (nullable) += the sufficient statistics of every sampled history
 * (_mjp.get_history_statistics, raoteh/sampler/_mjp.py:150).
 * Trajectories whose status != 0 are skipped; status 3 = more than `cap`
 * candidate events in one sweep, or more than 255 on one branch (the per-branch
 * counts are uint8; expected candidates per branch = omega * length) -- the
 * trajectory is left at its last completed sweep.
 */
int rt_raoteh_sweeps(int S, int n_nodes, int64_t n_traj, int64_t traj_stride, int64_t n_sites,
                     int64_t traj0, const int32_t* program, int n_ops, int n_slots,
                     const int32_t* parent, const double* length, const double* B,
                     const double* rate, const double* root_distn,
                     int obs_kind, const void* obs, int64_t obs_stride,
                     uint8_t* node_state, float* ev_time, uint8_t* ev_sb, uint8_t* ev_count,
                     int32_t* ev_total, int cap, uint64_t seed, int64_t sweep0, int n_sweeps,
                     int init_k, double* dwell_sum, double* trans_sum, int8_t* status,
                     void* stream);

/*
 * The same sweeps with the arguments in a struct, plus two options:
 *   time_f64    : every event time, branch position and Poisson hazard in fp64, the arithmetic of
 *                 the reference (raoteh/sampler/_sample_mjp.py:47-69 draws the event times with
 *                 numpy's fp64 exponentials); ev_time is then double [traj_stride][cap]
 *                 (S in {2,3,4,5,6,8}).  With 0, ev_time is float [traj_stride][cap] (half the
 *                 jump-list bytes).  Both consume the same Philox words in the same order.
 *   sweep_count : nullable int32 [traj_stride], the number of sweeps every trajectory has
 *                 completed.  When given, trajectory t runs sweeps sweep_count[t] .. sweep0 +
 *                 n_sweeps - 1 (Philox counter = its own sweep index) and the count is written
 *                 back, so a trajectory that stopped early (status 3, event capacity) can be
 *                 continued by repeating the call after growing `cap` and clearing its status:
 *                 every (trajectory, sweep) contributes to dwell_sum / trans_sum exactly once.
 */
typedef struct rt_raoteh_args {
  int32_t S, n_nodes, n_ops, n_slots, obs_kind, cap, n_sweeps, init_k;
  int32_t time_f64, reserved;
  int64_t n_traj, traj_stride, n_sites, traj0, obs_stride, sweep0;
  uint64_t seed;
  const int32_t* program;
  const int32_t* parent;
  const double* length;
  const double* B;
  const double* rate;
  const double* root_distn;
  const void* obs;
  uint8_t* node_state;
  void* ev_time;
  uint8_t* ev_sb;
  uint8_t* ev_count;
  int32_t* ev_total;
  int32_t* sweep_count;
  double* dwell_sum;
  double* trans_sum;
  int8_t* status;
} rt_raoteh_args;

int rt_raoteh_run(const rt_raoteh_args* args, void* stream);

/*
 * Exact posterior draws of whole histories (stochastic mapping; Nielsen 2002, Hobolth & Stone
 * 2009), one per trajectory, written in the trajectory layout of rt_raoteh_sweeps above, so that
 * rt_raoteh_run can continue from them.  The law drawn is the posterior of the MJP history given
 * the observations of the trajectory's site (site = (traj0 + t) % n_sites) -- the stationary law
 * of the sweeps, so a chain started from a draw needs no burn-in:
 *   node states  x_root ~ pi * L_root, then, walking the upward program backwards (parents first),
 *                x_c ~ P_c[x_a, :] * L_c with L_c the stored partial (OP_MSG_SLOT, store index =
 *                op field 3), the observation (OP_MSG_OBS) or ones (OP_MSG_ONES): the tree form of
 *                _sample_mc0.resample_states (raoteh/sampler/_sample_mc0.py:20);
 *   branch paths given (x_a, x_c, t_c), by uniformization with mu = max_s q_s, B = I + Q/mu:
 *                Pr(N = n) ~ Pois(n; mu t_c) (B^n)[x_a, x_c], intermediate states
 *                Pr(x_i = s) ~ B[x_{i-1}, s] (B^{N-i})[s, x_c], event times the order statistics
 *                of N uniforms on (0, t_c); only the state changes are stored, strictly inside
 *                (0, t_c) and strictly increasing in the stored precision.
 * It replaces the arbitrary initial history of _sampler.get_restricted_feasible_history
 * (raoteh/sampler/_sampler.py:563), which the sweeps must then forget.
 *
 * S in 2..8, observations RT_OBS_CODES or RT_OBS_MASK, fp64 event times (time_f64) except at
 * S = 7 (whose sweeps take float times only).  Inputs: program/parent/length as for the sweeps,
 * Q [S][S] with diagonal, P [n_nodes][S][S] = expm(t_b Q) (rt_expm_batched), partials and
 * site_status [n_sites] from rt_prune_loglik (site_stride = their row length), root_distn nullable.
 * The powers B^0..B^n_pow are built in a workspace, n_pow from the Poisson tail at
 * mu * max_b t_b, at most 320: a branch with mu * t_c beyond ~200 cannot be drawn (status 3;
 * subdivide it with degree-two nodes).
 * Philox4x32-10 keyed by (seed; traj0 + t, k): k is the draw's index in the chain's sweep
 * numbering (the draw uses its own substream, so a sweep with the same index draws other words);
 * results do not depend on how trajectories are split over launches or GPUs.
 * Outputs: the trajectory arrays; sweep_count (nullable) = k + 1 where the draw succeeded;
 * dwell_sum [S] / trans_sum [S*S] (nullable) += the statistics of the drawn histories.
 * status [traj_stride]: trajectories with status != 0 on entry are skipped; a trajectory whose
 * site has status != 0 gets that status; 1 = no feasible history, 3 = more than 255 real jumps on
 * a branch, a branch too long for the power table, or a jump time that cannot be stored,
 * 4 = more than `cap` real jumps in the trajectory (ev_total is then 0).
 */
typedef struct rt_posterior_draw_args {
  int32_t S, n_nodes, n_ops, cap, obs_kind, time_f64;
  int64_t n_traj, traj_stride, n_sites, traj0, obs_stride, site_stride;
  uint64_t seed;
  int64_t k;
  const int32_t* program;
  const int32_t* parent;
  const double* length;
  const double* Q;
  const double* P;
  const double* root_distn;
  const void* obs;
  const double* partials;
  const int8_t* site_status;
  uint8_t* node_state;
  void* ev_time;
  uint8_t* ev_sb;
  uint8_t* ev_count;
  int32_t* ev_total;
  int32_t* sweep_count;
  double* dwell_sum;
  double* trans_sum;
  int8_t* status;
} rt_posterior_draw_args;

int rt_posterior_draw(const rt_posterior_draw_args* args, void* stream);

/*
 * Exact posterior draws under a site-class mixture (+G rates, +I, per-class rate matrices): the
 * joint draw of (class, history) given the site's observations.  Each trajectory first draws its
 * site's class c from class_post[.][site] (the class posterior, e.g. w_k L_k / sum_j w_j L_j),
 * then the history exactly as rt_posterior_draw does, on class c's inputs.  Every field of `base`
 * means what it means for rt_posterior_draw, except:
 *   Q          [K][S][S], the class generators r_k Q_k (a rate-0 class has Q = 0: no jumps);
 *   P          [K][n_nodes][S][S], P_k = expm(t_b r_k Q_k) with t the tree lengths in `length`;
 *   partials   class k's stored partials at partials + k * partials_class_stride (doubles), each
 *              [n_store][S][site_stride];
 *   dwell_sum  [K][S] and trans_sum [K][S*S] += the statistics of the histories of each class;
 *              dwell and event times are in tree time;
 *   site_status  the mixture's (0 where some class is feasible);
 *   sweep_count  must be NULL (these draws are not a sweep of one MJP's chain).
 * class_post [K][class_post_stride] fp64, class_post_stride >= n_sites; site_class [traj_stride]
 * uint8: the class drawn for trajectory t (written where the site's status is 0).  1 <= K <= 255.
 * Philox4x32-10 keyed by (seed; traj0 + t, k) as in rt_posterior_draw: the class is drawn by the
 * rule of the node states (the first class of positive weight whose cumulative weight reaches
 * x = (u + 1/2) 2^-32 sum_k class_post) from u = word 0 of (substream 2, block 0); the history
 * uses substream 1 as in rt_posterior_draw, so with K = 1 it is bit for bit that draw.
 */
typedef struct rt_posterior_draw_mixture_args {
  rt_posterior_draw_args base;
  int32_t K, reserved;
  int64_t partials_class_stride, class_post_stride;
  const double* class_post;
  uint8_t* site_class;
} rt_posterior_draw_mixture_args;

int rt_posterior_draw_mixture(const rt_posterior_draw_mixture_args* args, void* stream);

/*
 * Forward (prior) simulation of n_traj independent sites: the batched replacement of the
 * reference's jump-by-jump simulator _sampler.get_forward_sample / gen_forward_samples
 * (raoteh/sampler/_sampler.py:67-235), one history per call there.  Trajectory t (0 <= t < n_traj)
 * is the global index traj0 + t; every output is written at t.
 *
 * Classes (site-class mixtures: +G rates, +I, per-class rate matrices), 1 <= K <= 255: the class c of
 * a site is drawn first from class_weight [K] (nullable when K = 1) and written to site_class
 * [traj_stride] (nullable).  Q [K][S][S] holds the class generators r_k Q_k (rate 0: Q = 0, an +I
 * class), P [K][n_nodes][S][S] their transition matrices expm(t_b r_k Q_k).  root_distn [S] is
 * nullable, and NULL means UNIFORM here (the pruning calls read NULL as weights of one); it is
 * normalised, as is every sampled row.  Both modes walk the upward program backwards (parents first):
 *   RT_SIM_NODES   x_root ~ pi, x_c ~ P_c[x_a, :] with negative round-off clamped to 0 and the row
 *                  renormalised (as synth.simulate_leaf_codes); P is read, Q and length are not.
 *   RT_SIM_HISTORY jump by jump on every branch as get_forward_sample: dwell ~ Exp(q_s) with
 *                  q_s = sum_{s' != s} Q[s][s'], next state ~ Q[s, :] / q_s.  The history is written
 *                  in the trajectory layout of rt_raoteh_run (node_state, ev_count, ev_total, ev_time,
 *                  ev_sb; jumps right-aligned at `cap`, upward-program order, child end first, times
 *                  strictly inside (0, t_b) and strictly increasing in the stored precision), so
 *                  rt_raoteh_run and rt_tmjp_run (RT_TMJP_TRAJ_LOGLIK) read it unchanged.  ev_time is
 *                  float, or double with time_f64.  dwell_sum [K][S] / trans_sum [K][S*S] (nullable,
 *                  together) += the statistics of the simulated histories; they are accumulated in
 *                  shared memory, K S (8 + 4 S) bytes, which must stay within 160 KiB.  Q and length
 *                  are read, P is not.
 *                  status [traj_stride] (required): 0, 3 = more than 255 jumps on one branch (the
 *                  uint8 counts; subdivide it with degree-two nodes) or a jump time that cannot be
 *                  stored, 4 = more than `cap` jumps in the trajectory (ev_total is then 0).  The node
 *                  states and leaf codes of such a site are still a draw from the prior.
 * node_state [n_nodes][traj_stride]: nullable in RT_SIM_NODES.
 * Leaf codes: obs (nullable) uint8 [n_slots][obs_stride] in the RT_OBS_CODES layout, obs_stride >=
 * n_traj; node v with obs_slot[v] >= 0 (obs_slot int32 [n_nodes]) writes its state to row obs_slot[v].
 * tmpl (nullable) uint8 [n_slots][tmpl_stride], the codes of a real alignment of tmpl_n_sites sites:
 * where tmpl[obs_slot[v]][(traj0 + t) % tmpl_n_sites] is RT_MISSING (255) the written code is too.
 * Randomness: Philox4x32-10 keyed by (seed; traj0 + t, k), k the replicate index, on its own
 * substream 0xffff (the sweeps use 0 and the warp kernel 0 .. (n_parts+2)(n_ops+1)-1 < 65535, the
 * exact draws 1 and 2): words 0 and 1 draw the class, words 2 and 3 seed the PCG32 stream of every
 * other draw.  Results do not depend on how sites are split over calls or GPUs.
 * Every draw reads one entry of a Walker alias table built per call (one per sampled row), so it is
 * O(1) for every S in 2..64; the tables take 4 bytes per entry: 4 K n_nodes S^2 (NODES) or 4 K S^2.
 */
#define RT_SIM_NODES 0
#define RT_SIM_HISTORY 1

typedef struct rt_forward_args {
  int32_t S, n_nodes, n_ops, K, mode, cap, time_f64, reserved;
  int64_t n_traj, traj_stride, traj0, obs_stride, tmpl_stride, tmpl_n_sites;
  uint64_t seed;
  int64_t k;
  const int32_t* program;      /* [n_ops][4] upward program (raoteh_b200/lowering.py) */
  const int32_t* parent;       /* [n_nodes] */
  const double* length;        /* [n_nodes] (HISTORY) */
  const int32_t* obs_slot;     /* [n_nodes], -1 = no leaf row (required with obs) */
  const double* class_weight;  /* [K] */
  const double* Q;             /* [K][S][S] (HISTORY) */
  const double* P;             /* [K][n_nodes][S][S] (NODES) */
  const double* root_distn;    /* [S], NULL = uniform */
  const uint8_t* tmpl;
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
} rt_forward_args;

int rt_forward_simulate(const rt_forward_args* args, void* stream);

/*
 * Warp-cooperative Rao-Teh kernels: one warp per (chain, site) trajectory.
 *
 * (1) Rao-Teh sweeps for S = 7 and 9 <= S <= 64 primary states (rt_raoteh_sweeps dispatches
 *     here; n_parts = 0): lanes own the states of the FFBS messages.
 * (2) The blocked Gibbs sampler of the compound TOLERANCE process
 *     (raoteh/sampler/_sample_tmjp_dense.py:40-171 gen_histories_v1,
 *     sparse twin _sample_tmjp.py:34-168): per sweep, Poisson events on the primary
 *     trajectory (:116-124), primary states given all tolerance trajectories with
 *     a chunk allowed iff none of its classes is ever off inside it
 *     (resample_primary_states_v1 :175-371), then for every tolerance class
 *     (lane = class) Poisson events (:146-155) and the 2-state FFBS with the class
 *     forced on wherever the primary state belongs to it, plus per-node disease
 *     data (resample_tolerance_states_v1 :374-506).  The merged trees and chunk
 *     trees of the reference (_graph_transform.add_trajectories :508,
 *     get_chunk_tree_type_b :298) are implicit in the per-edge event walk.
 *     mode RT_TMJP_INIT_PRIMARY / RT_TMJP_INIT_TOLERANCE build the initial
 *     feasible history (get_feasible_history :509-627: primary first, then one
 *     tolerance event at a uniform time inside every primary segment).
 * (3) The Rao-Blackwellised tolerance summary of a primary trajectory
 *     (raoteh/sampler/_tmjp_dense.py:724-855 get_tolerance_summary ->
 *     get_inhomogeneous_mjp :965, get_expected_tolerance_history_statistics :246,
 *     pyfelscore.get_tolerance_rate_matrix :239 / get_tolerance_expectations :339,
 *     closed forms raoteh/sampler/_linalg.py:14-118): lane = class, per segment
 *     the 2x2 block of expm(t Q3) and its Frechet integrals in closed form.
 *     mode RT_TMJP_SUMMARY, or flag RT_TMJP_F_SUMMARY after every sweep.
 *
 * Trajectory state, caller-owned device arrays:
 *   p_node/p_cnt uint8, element (trajectory t, node v) at t*pn_traj_stride + v*pn_node_stride
 *   p_total int32 [n_traj]; p_time float [n_traj][cap_p]; p_sb uint8 [n_traj][cap_p]
 *       (same jump-list convention as rt_raoteh_sweeps)
 *   t_node  uint32 [n_traj][n_nodes]          bit c = class c is ON at the node
 *   t_cnt   uint8  [n_traj][n_nodes][n_parts]  toggles of class c on the edge above the node
 *   t_total uint8  [n_traj][n_parts]
 *   t_time  float  [n_traj][n_parts][cap_t]    toggle times, same ordering convention
 * tol_obs (nullable): uint8 [n_tol_obs][n_parts][tol_obs_stride], bit0 = off allowed,
 *   bit1 = on allowed (the reference's disease_data); tol_obs_slot int32 [n_nodes], -1 = none.
 * status int8 [n_traj]: 0 ok, 1 infeasible (structural zero), 2 numerical zero in the
 *   summary, 3 event capacity exceeded in a sweep, 4 jump capacity exceeded, 6 no feasible
 *   tolerance history (disease data contradict the primary trajectory).
 * Outputs (all nullable, += over trajectories and sweeps): prim_dwell [S], prim_trans [S*S]
 *   (_mjp_dense.get_history_statistics, raoteh/sampler/_mjp_dense.py:150), tol_stats
 *   [n_parts][4] = (root on, dwell on, gains, losses) of the SAMPLED tolerance
 *   trajectories, summary_sum [8] = the 7 values of get_tolerance_summary (+ count);
 *   summary_out [n_traj][8] = the same per trajectory (last sweep), with [7] = the log-likelihood
 *   of the primary trajectory under the compound process with the tolerance histories integrated
 *   out (get_tolerance_process_log_likelihood, raoteh/sampler/_tmjp_dense.py:407-505).
 */
#define RT_TMJP_INIT_PRIMARY 0
#define RT_TMJP_INIT_TOLERANCE 1
#define RT_TMJP_SWEEP 2
#define RT_TMJP_SUMMARY 3
#define RT_TMJP_TRAJ_LOGLIK 4   /* traj_loglik[t] = log-likelihood of primary trajectory t under (B, omega_p, pi_p):
                                   _mjp.get_trajectory_log_likelihood, raoteh/sampler/_mjp.py:186-250; with
                                   RT_TMJP_F_STATS_PRIMARY also prim_dwell / prim_trans += the statistics of the
                                   CURRENT histories (_mjp_dense.get_history_statistics :150) */
#define RT_TMJP_F_STATS_PRIMARY 1
#define RT_TMJP_F_STATS_TOLERANCE 2
#define RT_TMJP_F_SUMMARY 4
#define RT_TMJP_F_SKIP_PRIMARY 8    /* sweep: tolerance half only (phase-split launches) */
#define RT_TMJP_F_SKIP_TOLERANCE 16 /* sweep: primary half only */

typedef struct rt_tmjp_args {
  /* model and tree */
  int32_t S, n_parts, n_nodes, n_ops, n_slots;
  int32_t cap_p, cap_t, obs_kind;
  const int32_t* program;      /* [n_ops][4] upward program */
  const int32_t* parent;       /* [n_nodes] */
  const double* length;        /* [n_nodes] */
  const double* B;             /* [S][S] I + Q_primary/omega_p */
  const double* rate_p;        /* [S] omega_p - q_s */
  const double* pi_p;          /* [S] primary root distribution, NULL = ones */
  const uint8_t* part;         /* [S] tolerance class of a primary state (n_parts > 0) */
  const double* absorb;        /* [S][n_parts] sum of Q[s,s'] over s' != s in class c */
  double rate_on, rate_off, omega_t;
  double omega_p;              /* primary uniformization rate (Q[a][b] = omega_p * B[a][b], a != b) */
  /* observations */
  const void* obs;             /* primary: codes or masks per site */
  int64_t obs_stride;
  const uint8_t* tol_obs;
  const int32_t* tol_obs_slot;
  int64_t tol_obs_stride;
  /* trajectories */
  int64_t n_traj, n_sites, traj0;
  uint8_t* p_node;
  uint8_t* p_cnt;
  int64_t pn_traj_stride, pn_node_stride;
  int32_t* p_total;
  float* p_time;
  uint8_t* p_sb;
  uint32_t* t_node;
  uint8_t* t_cnt;
  uint8_t* t_total;
  float* t_time;
  int8_t* status;
  /* control */
  uint64_t seed;
  int64_t sweep0;
  int32_t n_sweeps, mode, init_k, flags;
  /* outputs */
  double* prim_dwell;
  double* prim_trans;
  double* tol_stats;
  double* summary_sum;
  double* summary_out;
  double* traj_loglik;         /* [n_traj], mode RT_TMJP_TRAJ_LOGLIK */
  const double* p_time64;      /* nullable [n_traj][cap_p]: fp64 jump times of caller-loaded primary
                                  trajectories (same layout as p_time); modes SUMMARY / TRAJ_LOGLIK then
                                  use them, and the fp64 branch lengths, instead of the float32 state */
} rt_tmjp_args;

int rt_tmjp_run(const rt_tmjp_args* args, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RT_B200_H */
