// K4/K5 for small state spaces (S <= 8): downward pass, posterior node
// marginals and per-edge sufficient statistics, batched over sites.
//
// Replaces, batched over sites,
//   pyfelscore.mc0_esd_get_node_to_distn       (raoteh/sampler/_mc0_dense.py:381,
//        _mcy_dense.py:195; spec _mc0_dense.py:400-489)
//   pyfelscore.mc0_esd_get_joint_endpoint_distn (_mcy_dense.py:205; spec
//        _mc0_dense.py:217-270)
// and the `joint_prob / cond_prob` accumulation of
//   _mjp_dense.get_expected_history_statistics  (_mjp_dense.py:502-510,521-533).
//
// Edge-major and level-synchronous: one launch per tree level, grid =
// (site chunks) x (edges of the level).  A thread strides over the sites of its
// chunk, so the S*S weights W_b += G_b (x) L_b accumulate in registers with no
// cross-lane traffic until one block reduction + S*S atomics per CTA.  The
// joint J_b = G_b[:,None] * P_b * L_b[None,:] is never materialised.
// HBM traffic per site and edge: D_parent in, L_child in, D_child out
// (3 * S * 8 B; leaves read 1 code byte instead) -- HBM-bound.
#include <type_traits>

#include "rt_common.cuh"

namespace {

constexpr int kBlock = 256;
constexpr int kSitesPerCta = 2048;

// site_weight (nullable): D[root] = w_site * norm(pi o L_root).  The level kernels below only
// propagate the root marginal, so every marginal and W of the site then carries the weight.
template <int S>
__global__ void __launch_bounds__(kBlock)
root_distn_kernel(int64_t n_sites, int64_t stride, int64_t nd_stride, const double* __restrict__ root_distn,
                  const double* __restrict__ partials, const int8_t* __restrict__ status,
                  const double* __restrict__ site_weight, double* __restrict__ node_distn,
                  double* __restrict__ root_post_sum) {
  __shared__ double red[kBlock / 32][S];
  const int tid = threadIdx.x;
  double sum[S];
#pragma unroll
  for (int s = 0; s < S; ++s) sum[s] = 0.0;
  for (int64_t site = (int64_t)blockIdx.x * kBlock + tid; site < n_sites;
       site += (int64_t)gridDim.x * kBlock) {
    if (status[site] != RT_SITE_OK) {
#pragma unroll
      for (int s = 0; s < S; ++s) node_distn[(int64_t)s * nd_stride + site] = 0.0;
      continue;
    }
    double w[S];
    double tot = 0.0;
#pragma unroll
    for (int s = 0; s < S; ++s) {
      w[s] = partials[(int64_t)s * stride + site] * (root_distn ? root_distn[s] : 1.0);
      tot += w[s];
    }
    const double inv = (site_weight ? site_weight[site] : 1.0) / tot;
#pragma unroll
    for (int s = 0; s < S; ++s) {
      const double d = w[s] * inv;
      node_distn[(int64_t)s * nd_stride + site] = d;
      sum[s] += d;
    }
  }
  if (root_post_sum) {
#pragma unroll
    for (int s = 0; s < S; ++s) {
      double v = rt_warp_sum(sum[s]);
      if ((tid & 31) == 0) red[tid >> 5][s] = v;
    }
    __syncthreads();
    if (tid < S) {
      double t = 0.0;
      for (int i = 0; i < kBlock / 32; ++i) t += red[i][tid];
      atomicAdd(&root_post_sum[tid], t);
    }
  }
}

// PACKED: RT_OBS_CODES4 leaf codes.  BR: also the per-site branch expectation of the walk's BR.
// Node marginals are indexed with their own site stride (a workspace holds only this chunk).
template <int S, int OBS, bool BR, bool PACKED>
__global__ void __launch_bounds__(kBlock)
down_level_kernel(int64_t n_sites, int64_t stride, int64_t nd_stride, const int4* __restrict__ edges,
                  const double* __restrict__ P, const void* __restrict__ obs,
                  const double* __restrict__ partials, const int8_t* __restrict__ status,
                  double* __restrict__ node_distn, double* __restrict__ W,
                  const double* __restrict__ Kmat, double* __restrict__ branch_out) {
  __shared__ double Ps[S * S];
  __shared__ double Ks[BR ? S * S : 1];
  __shared__ double red[kBlock / 32][S * S];
  const int tid = threadIdx.x;
  const int4 e = edges[blockIdx.y];   // (child node, parent store, child store, child obs slot)
  const int b = e.x;
  if (tid < S * S) Ps[tid] = P[(size_t)b * S * S + tid];
  if (BR && tid < S * S) Ks[tid] = Kmat[(size_t)b * S * S + tid];
  __syncthreads();

  double Wacc[S][S];
#pragma unroll
  for (int i = 0; i < S; ++i)
#pragma unroll
    for (int j = 0; j < S; ++j) Wacc[i][j] = 0.0;

  const double* Dp = node_distn + (int64_t)e.y * S * nd_stride;
  const double* Lc = e.z >= 0 ? partials + (int64_t)e.z * S * stride : nullptr;
  double* Dc = e.z >= 0 ? node_distn + (int64_t)e.z * S * nd_stride : nullptr;

  const int64_t lo = (int64_t)blockIdx.x * kSitesPerCta;
  const int64_t hi = (n_sites < lo + kSitesPerCta) ? n_sites : lo + kSitesPerCta;

  // loads of one site (software-pipelined: the next site's loads are in flight
  // while the current one is computed)
  auto load_site = [&](int64_t site, double (&L)[S], double (&D)[S], bool& ok) {
    ok = site < hi && status[site] == RT_SITE_OK;
    if (!ok) {
#pragma unroll
      for (int s = 0; s < S; ++s) { L[s] = 0.0; D[s] = 0.0; }
      return;
    }
    if (Lc) {
#pragma unroll
      for (int s = 0; s < S; ++s) L[s] = __ldcs(&Lc[(int64_t)s * stride + site]);
    } else if (e.w < 0) {
#pragma unroll
      for (int s = 0; s < S; ++s) L[s] = 1.0;
    } else if (OBS == OBS_CODES) {
      const uint8_t* row = reinterpret_cast<const uint8_t*>(obs);
      int k;
      if (PACKED) {      // nibble site & 1 of byte site >> 1, 15 = unobserved
        k = (row[(int64_t)e.w * ((stride + 1) >> 1) + (site >> 1)] >> ((int)(site & 1) * 4)) & 15;
        if (k == 15) k = RT_MISSING;
      } else {
        k = row[(int64_t)e.w * stride + site];
      }
#pragma unroll
      for (int s = 0; s < S; ++s) L[s] = (k == RT_MISSING || k == s) ? 1.0 : 0.0;
    } else if (OBS == OBS_MASK) {
      const unsigned long long mk =
          reinterpret_cast<const unsigned long long*>(obs)[(int64_t)e.w * stride + site];
#pragma unroll
      for (int s = 0; s < S; ++s) L[s] = ((mk >> s) & 1ull) ? 1.0 : 0.0;
    } else {
      const double* d = reinterpret_cast<const double*>(obs);
#pragma unroll
      for (int s = 0; s < S; ++s) L[s] = d[((int64_t)e.w * S + s) * stride + site];
    }
#pragma unroll
    for (int s = 0; s < S; ++s) D[s] = Dp[(int64_t)s * nd_stride + site];
  };

  // P_b is re-read from shared memory at every use from S = 7 on: kept in registers across the
  // site loop (S * S values), it and the S x S accumulator would not fit in 255 registers
  auto p_at = [&](int i) -> double {
    if constexpr (S >= 7) return reinterpret_cast<volatile const double*>(Ps)[i];
    else return Ps[i];
  };
  // the next site's loads are issued before the current site is computed up to S = 5; from S = 6
  // on, their 2 S registers next to the S x S accumulator would spill
  constexpr bool kPrefetch = S <= 5;
  double Ln[S], Dn[S];
  bool okn = false;
  if (kPrefetch) load_site(lo + tid, Ln, Dn, okn);
  for (int64_t site = lo + tid; site < hi; site += kBlock) {
    double L[S], D[S];
    bool ok;
    if (kPrefetch) {
      ok = okn;
#pragma unroll
      for (int s = 0; s < S; ++s) { L[s] = Ln[s]; D[s] = Dn[s]; }
      load_site(site + kBlock, Ln, Dn, okn);
    } else {
      load_site(site, L, D, ok);
    }
    if (!ok) {
      if (Dc) {
#pragma unroll
        for (int s = 0; s < S; ++s) Dc[(int64_t)s * nd_stride + site] = 0.0;
      }
      if (BR) branch_out[(int64_t)b * stride + site] = 0.0;
      continue;
    }
    double G[S];
#pragma unroll
    for (int a = 0; a < S; ++a) {
      double m = 0.0;
#pragma unroll
      for (int c = 0; c < S; ++c) m = fma(p_at(a * S + c), L[c], m);
      G[a] = (D[a] > 0.0) ? D[a] / m : 0.0;
    }
    if (Dc) {
#pragma unroll
      for (int c = 0; c < S; ++c) {
        double t = 0.0;
#pragma unroll
        for (int a = 0; a < S; ++a) t = fma(G[a], p_at(a * S + c), t);
        Dc[(int64_t)c * nd_stride + site] = t * L[c];
      }
    }
    if (BR) {
      double x = 0.0;
#pragma unroll
      for (int a = 0; a < S; ++a) {
        double kl = 0.0;
#pragma unroll
        for (int c = 0; c < S; ++c) kl = fma(Ks[a * S + c], L[c], kl);
        x = fma(G[a], kl, x);
      }
      branch_out[(int64_t)b * stride + site] = x;
    }
#pragma unroll
    for (int a = 0; a < S; ++a)
#pragma unroll
      for (int c = 0; c < S; ++c) Wacc[a][c] = fma(G[a], L[c], Wacc[a][c]);
  }

#pragma unroll
  for (int a = 0; a < S; ++a)
#pragma unroll
    for (int c = 0; c < S; ++c) {
      double v = rt_warp_sum(Wacc[a][c]);
      if ((tid & 31) == 0) red[tid >> 5][a * S + c] = v;
    }
  __syncthreads();
  if (tid < S * S) {
    double t = 0.0;
    for (int i = 0; i < kBlock / 32; ++i) t += red[i][tid];
    if (Ps[tid] > 0.0 && t != 0.0) atomicAdd(&W[(size_t)b * S * S + tid], t);
  }
}

template <int S, int OBS, bool BR, bool PACKED>
void launch_levels(int64_t n_sites, int64_t stride, int64_t nd_stride, const int4* edges,
                   const int32_t* level_ptr_h, int n_levels, const double* P, const void* obs,
                   const double* partials, const int8_t* status, double* node_distn, double* W,
                   const double* Kmat, double* branch_out, cudaStream_t stream) {
  const unsigned gx = (unsigned)((n_sites + kSitesPerCta - 1) / kSitesPerCta);
  for (int l = 0; l < n_levels; ++l) {
    const int e0 = level_ptr_h[l], e1 = level_ptr_h[l + 1];
    if (e1 <= e0) continue;
    dim3 grid(gx, (unsigned)(e1 - e0));
    down_level_kernel<S, OBS, BR, PACKED><<<grid, kBlock, 0, stream>>>(
        n_sites, stride, nd_stride, edges + e0, P, obs, partials, status, node_distn, W, Kmat,
        branch_out);
  }
}


// ---------------------------------------------------------------------------------------
// Fused downward WALK: one thread per site runs the whole downward pass by walking the
// upward program backwards (same slot assignment, liveness reversed), with the current
// node marginal in registers and parked marginals in a per-thread shared-memory stack.
// Nothing but the stored partials is read from HBM and node marginals are written only on
// request.  The per-edge weights W_b += G (x) L are reduced across the warp with a
// transpose (reduce-scatter) butterfly -- V = S*S values over 32 lanes in
// V/2 + V/4 + ... exchanges instead of V full reductions -- and then added to a per-CTA
// accumulator in shared memory; one masked global atomicAdd per entry per CTA at the end.
//
// Lane frames (S = 4): lane l holds every S-vector with its states permuted by an XOR mask,
// a parent-side vector (the node marginal `cur`, G) in frame x = (l >> 3) & 3 -- element a is
// state a ^ x -- and a child-side vector (L, the child marginal t) in frame y = (l >> 1) & 3.
// Entry (a, b) of G (x) L then sits in register ((a ^ x) << 2) | (b ^ y) = (4a + b) ^ z with
// z = (l >> 1) & 15, and in every stage of the butterfly the lane keeps the lower half of its
// registers and sends the upper half: the stages are shuffles and adds without selects (two
// FSEL per double and per half before).  The frame costs per-lane addresses: P, K and the leaf
// reciprocal table are read at permuted indices, stored partials at row b ^ y, node marginals
// are written to rows a ^ x / b ^ y, and a child marginal goes to the stack at position
// b ^ x ^ y, so that it reads back in frame x -- also the one the next op consumes, which
// otherwise stays in registers (the round trip costs fewer instructions than 16 FSEL per site).
// Only the S = 4 kernels without per-branch output use frames: with them, the per-branch
// kernel needed 75 more registers (233) and lost a CTA per SM.  Elsewhere both masks are 0.
// ---------------------------------------------------------------------------------------
#ifndef RT_WALK_BLOCK
#define RT_WALK_BLOCK 128
#endif
// G = D / m: D == 0 gives 0 * (1/m) = 0 for any m > 0, so only m > 0 needs a test (one DSETP
// per entry less on the FP64 pipe); RT_WALK_TEST_D=1 restores the explicit D > 0 test
#ifndef RT_WALK_TEST_D
#define RT_WALK_TEST_D 0
#endif
#if RT_WALK_TEST_D
#define RT_WALK_DCHECK(d) (d) > 0.0 &&
#else
#define RT_WALK_DCHECK(d)
#endif
#ifndef RT_WALK_L2PF
#define RT_WALK_L2PF 0      // distance (ops) of the extra L2 prefetch of stored partials; 0 = off
#endif
constexpr int kWalkBlock = RT_WALK_BLOCK;

// FRAMED: the lane's values are in the lane frame described above (V = 16), so that the lane
// keeps v[i] and sends v[i + half] in every stage; otherwise it picks the halves by its lane bit
template <int V, bool FRAMED>
__device__ __forceinline__ void reduce_scatter_warp(double (&v)[V], int lane) {
  // after the call: V==16 -> lane holds value (lane>>1) in v[0]; V==32 -> value `lane`;
  // V==64 -> values 2*lane, 2*lane+1 in v[0], v[1]   (all fully summed over the warp)
  int len = V;
#pragma unroll
  for (int m = 16; m >= 1; m >>= 1) {
    if (len > 1) {
      const bool up = !FRAMED && (lane & m) != 0;
      const int half = len / 2;
#pragma unroll
      for (int i = 0; i < V / 2; ++i) {
        if (i < half) {
          const double send = up ? v[i] : v[i + half];
          const double keep = up ? v[i + half] : v[i];
          v[i] = keep + __shfl_xor_sync(0xffffffffu, send, m);
        }
      }
      len = half;
    } else {
      v[0] += __shfl_xor_sync(0xffffffffu, v[0], m);
    }
  }
}

template <int S> struct WalkV { static constexpr int value = (S <= 4) ? 16 : (S == 5 ? 32 : 64); };

// v[i] <- v[i ^ d] for a 2-bit lane mask d (S = 4): two select stages
__device__ __forceinline__ void xor_permute4(double (&v)[4], int d) {
  const bool b0 = (d & 1) != 0, b1 = (d & 2) != 0;
  double u[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) u[i] = b0 ? v[i ^ 1] : v[i];
#pragma unroll
  for (int i = 0; i < 4; ++i) v[i] = b1 ? u[i ^ 2] : u[i];
}
// sites per thread: more sites amortise the per-op work (program decode, P loads, the
// cross-lane reduction of W) over more arithmetic; bounded by registers
#ifndef RT_WALK_NS
#define RT_WALK_NS 2
#endif
template <int S> struct WalkNS { static constexpr int value = (S <= 4) ? RT_WALK_NS : 2; };

// 1/x to ~1 ulp: hardware seed (rcp.approx.ftz.f64, ~20 bits, full double range) plus two
// Newton steps.  Replaces the ~20-instruction IEEE division; the quotient is within 2 ulp,
// far inside the 1e-10 tolerance of the path.
__device__ __forceinline__ double fast_rcp(double x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  r = r * fma(-x, r, 2.0);
  r = r * fma(-x, r, 2.0);
  return r;
}

// BR: also write, per site and branch, x = sum_ab G_a K_b[a,c] L_c -- the posterior expectation
// of the statistic whose per-edge kernel is K (e.g. K_b = L(t_b Q, t_b (E o Q)): expected number
// of E-type transitions on the branch, examples/code2x3/extras.py:19-132).
// WEIGHTED: the root marginal of a site is w_site * norm(pi o L_root) (site_weight[n_sites]).
// Nothing below the root renormalises, so W, root_post_sum and the node marginals carry the
// weight.  site_weight is the last parameter: the WEIGHTED = false instantiations never read it
// and keep the parameter layout of the kernel without it.  With a minimum of one CTA per SM
// (none for the unweighted kernels, as before) ptxas gives the weighted walk the registers it
// needs: with the default heuristic it spilled 4-20 bytes for S = 2..4, and with this none up to
// S = 6.
template <int S, int OBS, bool BR, bool PACKED, bool WEIGHTED>
__global__ void __launch_bounds__(kWalkBlock, WEIGHTED ? 1 : (S == 4 && !BR ? 4 : 0))
down_walk_kernel(int64_t n_sites, int64_t stride, const int4* __restrict__ program, int n_ops,
                 int n_slots, int n_nodes, const double* __restrict__ P,
                 const double* __restrict__ root_distn, const void* __restrict__ obs,
                 const double* __restrict__ partials, const int8_t* __restrict__ status,
                 double* __restrict__ node_distn, double* __restrict__ W,
                 double* __restrict__ root_post_sum, const double* __restrict__ Kmat,
                 double* __restrict__ branch_out, const double* __restrict__ site_weight) {
  constexpr int obs_packed = PACKED ? 1 : 0;   // RT_OBS_CODES4 decoded at compile time
  constexpr int V = WalkV<S>::value;
  constexpr int NS = WalkNS<S>::value;
  constexpr int SP1 = S + 1;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  int4* prog_s = reinterpret_cast<int4*>(smem_raw);
  long long* off_s = reinterpret_cast<long long*>(prog_s + n_ops);   // [n_ops] element offset of the op's rows
  double* pi_s = reinterpret_cast<double*>(off_s + n_ops);
  double* P_s = pi_s + S;                              // [n_nodes][S][S]
  double* Pl_s = P_s + (size_t)n_nodes * S * S;        // [n_nodes][S][S+1]: RECIPROCALS of the columns and of the row sum (leaf edges)
  double* W_s = Pl_s + (size_t)n_nodes * S * SP1;      // [n_nodes][S*S] per-CTA accumulator
  double* rp_s = W_s + (size_t)n_nodes * S * S;        // [S]
  double* K_s = rp_s + S;                              // [n_nodes][S][S] (BR only)
  double* stk = K_s + (BR ? (size_t)n_nodes * S * S : 0);   // [n_slots][NS][S][kWalkBlock]

  const int tid = threadIdx.x, lane = tid & 31;
  for (int i = tid; i < n_ops; i += kWalkBlock) {
    const int4 op = program[i];
    prog_s[i] = op;
    const int code = op.x & 0xff;
    long long off = 0;
    if (code == OP_MSG_SLOT || code == OP_ROOT) off = (long long)op.w * S * stride;
    else if (code == OP_MSG_OBS)
      off = (OBS == OBS_DENSE) ? (long long)op.z * S * stride
                               : (long long)op.z * (obs_packed ? ((stride + 1) >> 1) : stride);
    off_s[i] = off;
  }
  if (tid < S) { pi_s[tid] = root_distn ? root_distn[tid] : 1.0; rp_s[tid] = 0.0; }
  for (int i = tid; i < n_nodes * S * S; i += kWalkBlock) { P_s[i] = P[i]; W_s[i] = 0.0; }
  if (BR)
    for (int i = tid; i < n_nodes * S * S; i += kWalkBlock) K_s[i] = Kmat[i];
  for (int i = tid; i < n_nodes * S; i += kWalkBlock) {
    double t = 0.0;
#pragma unroll
    for (int b = 0; b < S; ++b) {
      const double v = P[(size_t)i * S + b];
      Pl_s[i * SP1 + b] = v > 0.0 ? 1.0 / v : 0.0;     // 0 keeps G = 0 where the message is 0
      t += v;
    }
    Pl_s[i * SP1 + S] = t > 0.0 ? 1.0 / t : 0.0;
  }
  __syncthreads();

  // lane frames (see the header of the walk): parent side x, child side y, W register z
  constexpr bool kFramed = S == 4 && !BR;
  const int fx = kFramed ? (lane >> 3) & 3 : 0;
  const int fy = kFramed ? (lane >> 1) & 3 : 0;
  const int fz = (fx << 2) | fy;     // P'[a][b] = P[a ^ x][b ^ y] = P[(4a + b) ^ z] for S = 4
  const int fd = fx ^ fy;            // child frame -> parent frame
  static_assert(!kFramed || (kWalkBlock & (kWalkBlock - 1)) == 0, "stack rows are XOR-addressed");
  // entry i of the S x S table of node c (P_s) in the lane's frame.  Framed, a table is 128
  // bytes, so the permuted byte offset is one XOR (LOP3) with the lane part folded into `cz`.
  auto tab = [&](const double* t, int c, int i) -> double {
    if constexpr (kFramed) {
      const unsigned cz = (unsigned)c * (S * S * 8) | (unsigned)fz * 8;
      return *reinterpret_cast<const double*>(reinterpret_cast<const char*>(t) + (cz ^ (unsigned)(i * 8)));
    } else {
      return t[c * S * S + i];
    }
  };
  const int64_t tile_sites = (int64_t)kWalkBlock * NS;
  // framed: a 32-bit tile index, and the thread index read again at the end, keep the kernels at
  // 128 registers (4 CTAs per SM) without spills
  using TileIdx = typename std::conditional<kFramed, int, int64_t>::type;
  const TileIdx tiles = (TileIdx)((n_sites + tile_sites - 1) / tile_sites);
  for (TileIdx tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const int64_t site0 = (int64_t)tile * tile_sites + tid;            // site of q: site0 + q*kWalkBlock
    // the NEXT tile's leaf-code rows: pulled into L2 a whole tile ahead (the byte loads one op ahead
    // of their use cannot hide a DRAM round trip behind a short leaf op: 9 % of the warp samples
    // sat on that load, ncu source view)
    if (OBS == OBS_CODES && tile + gridDim.x < tiles) {
      const int64_t row_bytes = obs_packed ? tile_sites / 2 : tile_sites;
      const int lines_per_row = (int)((row_bytes + 127) / 128);
      const int64_t nb = (tile + gridDim.x) * row_bytes;
      for (int i = tid; i < n_ops * lines_per_row; i += kWalkBlock) {
        const int4 px = prog_s[i / lines_per_row];
        if ((px.x & 0xff) == OP_MSG_OBS)
          asm volatile("prefetch.global.L2 [%0];" :: "l"(reinterpret_cast<const uint8_t*>(obs) +
                       off_s[i / lines_per_row] + nb + (i % lines_per_row) * 128));
      }
    }
    bool live[NS];
#pragma unroll
    for (int q = 0; q < NS; ++q) {
      const int64_t site = site0 + q * kWalkBlock;
      live[q] = site < n_sites && status[site] == RT_SITE_OK;
    }
    double cur[NS][S];
#pragma unroll
    for (int q = 0; q < NS; ++q)
#pragma unroll
      for (int s = 0; s < S; ++s) cur[q][s] = 0.0;

    // The walk of one site is a serial chain, so the loads of op ip-1 (stored partial of an
    // internal child, or the code byte of a leaf) are issued into a second register buffer
    // before op ip is computed: ping-pong buffers, loop unrolled by two.
    auto issue = [&](int j, double (&Lb)[NS][S], int (&kb)[NS]) {
#if RT_WALK_L2PF > 0
      // stored partials of the op RT_WALK_L2PF further down the walk: pulled into L2 now, so the
      // register prefetch one op ahead of the use finds them there
      if (j - RT_WALK_L2PF >= 0) {
        const int4 px = prog_s[j - RT_WALK_L2PF];
        if ((px.x & 0xff) == OP_MSG_SLOT) {
          const double* src = partials + off_s[j - RT_WALK_L2PF] + site0;
#pragma unroll
          for (int q = 0; q < NS; ++q)
#pragma unroll
            for (int s = 0; s < S; ++s)
              asm volatile("prefetch.global.L2 [%0];" :: "l"(src + (int64_t)s * stride + q * kWalkBlock));
        }
      }
#endif
      if (j < 0) return;
      const int4 nx = prog_s[j];
      const int ncode = nx.x & 0xff;
      if (ncode == OP_MSG_SLOT) {
        const double* src = partials + off_s[j] + site0;
#pragma unroll
        for (int q = 0; q < NS; ++q)
#pragma unroll
          for (int s = 0; s < S; ++s)
            Lb[q][s] = live[q] ? __ldcs(&src[(int64_t)(s ^ fy) * stride + q * kWalkBlock]) : 0.0;
      } else if (ncode == OP_MSG_OBS && OBS == OBS_CODES) {
        const uint8_t* row = reinterpret_cast<const uint8_t*>(obs) + off_s[j];
#pragma unroll
        for (int q = 0; q < NS; ++q) {
          const int64_t sg = site0 + q * kWalkBlock;
          int k = 0;
          if (live[q]) {
            if (obs_packed) {      // RT_OBS_CODES4: nibble sg & 1 of byte sg >> 1, 15 = unobserved
              k = (row[sg >> 1] >> ((int)(sg & 1) * 4)) & 15;
              if (k == 15) k = RT_MISSING;
            } else {
              k = row[sg];
            }
          }
          kb[q] = k;
        }
      }
    };
    auto do_op = [&](int ip, const double (&Lb)[NS][S], const int (&kb)[NS]) {
      const int4 op = prog_s[ip];
      const int code = op.x & 0xff;
      if (code == OP_ROOT) {
        const double* src = partials + off_s[ip] + site0;
#pragma unroll
        for (int q = 0; q < NS; ++q) {
          double tot = 0.0;
#pragma unroll
          for (int s = 0; s < S; ++s) {
            cur[q][s] = live[q] ? src[(int64_t)(s ^ fx) * stride + q * kWalkBlock] * pi_s[s ^ fx] : 0.0;
            tot += cur[q][s];
          }
          const double num = WEIGHTED ? (live[q] ? site_weight[site0 + q * kWalkBlock] : 0.0) : 1.0;
          const double inv = tot > 0.0 ? num / tot : 0.0;
#pragma unroll
          for (int s = 0; s < S; ++s) {
            cur[q][s] *= inv;
            if (node_distn && site0 + q * kWalkBlock < n_sites)
              node_distn[off_s[ip] + (int64_t)(s ^ fx) * stride + site0 + q * kWalkBlock] = cur[q][s];
          }
        }
        if (root_post_sum) {
          double ts[S];
#pragma unroll
          for (int s = 0; s < S; ++s) {
            ts[s] = 0.0;
#pragma unroll
            for (int q = 0; q < NS; ++q) ts[s] += cur[q][s];
          }
          if constexpr (kFramed) xor_permute4(ts, fx);     // back to the natural state order
#pragma unroll
          for (int s = 0; s < S; ++s) {
            const double t = rt_warp_sum(ts[s]);
            if (lane == 0 && t != 0.0) atomicAdd(&rp_s[s], t);
          }
        }
      } else if (code == OP_STORE) {
        // a marginal parked by a non-fresh OP_MSG_SLOT (a fresh one is still in `cur`)
        if (op.x & OP_FLAG_PARK) {
#pragma unroll
          for (int q = 0; q < NS; ++q)
#pragma unroll
            for (int s = 0; s < S; ++s) cur[q][s] = stk[((op.z * NS + q) * S + s) * kWalkBlock + tid];
        }
      } else if (code <= OP_MSG_ONES) {
        const int c = op.y;
        double w[V];
#pragma unroll
        for (int i = 0; i < V; ++i) w[i] = 0.0;
        if (code == OP_MSG_SLOT) {
          // ---- internal child: its marginal D_c = L o (P^T G) is parked (or kept) ----
          double Pr[S * S];
#pragma unroll
          for (int i = 0; i < S * S; ++i) Pr[i] = tab(P_s, c, i);
          const bool fresh = (op.x & OP_FLAG_FRESH) != 0;   // next (reverse) op is the child's OP_STORE
#pragma unroll
          for (int q = 0; q < NS; ++q) {
            double L[S];
#pragma unroll
            for (int s = 0; s < S; ++s) L[s] = Lb[q][s];
            double G[S];
#pragma unroll
            for (int a = 0; a < S; ++a) {
              double m = 0.0;
#pragma unroll
              for (int b = 0; b < S; ++b) m = fma(Pr[a * S + b], L[b], m);
              G[a] = (RT_WALK_DCHECK(cur[q][a]) m > 0.0) ? cur[q][a] * fast_rcp(m) : 0.0;
            }
            double t[S];
#pragma unroll
            for (int b = 0; b < S; ++b) {
              double acc = 0.0;
#pragma unroll
              for (int a = 0; a < S; ++a) acc = fma(G[a], Pr[a * S + b], acc);
              t[b] = acc * L[b];
            }
#pragma unroll
            for (int i = 0; i < S * S; ++i) w[i] = fma(G[i / S], L[i % S], w[i]);
            if (BR) {
              double x = 0.0;
#pragma unroll
              for (int a = 0; a < S; ++a) {
                double kl = 0.0;
#pragma unroll
                for (int b = 0; b < S; ++b) kl = fma(K_s[c * S * S + a * S + b], L[b], kl);
                x = fma(G[a], kl, x);
              }
              if (site0 + q * kWalkBlock < n_sites) branch_out[(int64_t)c * stride + site0 + q * kWalkBlock] = x;
            }
#pragma unroll
            for (int b = 0; b < S; ++b) {
              // framed: position b ^ x ^ y, as one XOR of the row index (S * kWalkBlock is a power of 2)
              const int pos = kFramed ? ((((op.z * NS + q) * S * kWalkBlock) | (fd * kWalkBlock + tid)) ^ (b * kWalkBlock))
                                      : ((op.z * NS + q) * S + b) * kWalkBlock + tid;
              if (!fresh || kFramed) stk[pos] = t[b];
              if (node_distn && site0 + q * kWalkBlock < n_sites)
                node_distn[off_s[ip] + (int64_t)(b ^ fy) * stride + site0 + q * kWalkBlock] = t[b];
            }
            if (fresh) {
#pragma unroll
              for (int b = 0; b < S; ++b) cur[q][b] = kFramed ? stk[((op.z * NS + q) * S + b) * kWalkBlock + tid] : t[b];
            }
          }
        } else if (code == OP_MSG_OBS && OBS == OBS_CODES) {
          // ---- observed leaf, hard code k: P L is column k of P (the row sum when missing), so
          // G = D / (P L) is a product with an entry of a per-edge reciprocal table: no division
          // per site (the reciprocals were 6 % of the instructions of the walk, ncu source view)
          const double* Pl = Pl_s + c * S * SP1;
#pragma unroll
          for (int q = 0; q < NS; ++q) {
            const int k = kb[q];
            const int col = k == RT_MISSING ? S : k;
            double G[S], L[S];
#pragma unroll
            for (int a = 0; a < S; ++a) {
              G[a] = cur[q][a] * Pl[(a ^ fx) * SP1 + col];     // (a site that failed carries D = 0 from the root op)
              L[a] = (k == RT_MISSING || (k ^ fy) == a) ? 1.0 : 0.0;
            }
#pragma unroll
            for (int i = 0; i < S * S; ++i) w[i] = fma(G[i / S], L[i % S], w[i]);
            if (BR) {
              double x = 0.0;
#pragma unroll
              for (int a = 0; a < S; ++a) {
                double kl = 0.0;
#pragma unroll
                for (int b = 0; b < S; ++b) kl = fma(K_s[c * S * S + a * S + b], L[b], kl);
                x = fma(G[a], kl, x);
              }
              if (site0 + q * kWalkBlock < n_sites) branch_out[(int64_t)c * stride + site0 + q * kWalkBlock] = x;
            }
          }
        } else {
          // ---- leaf with a mask / dense emission row / no observation ----
          double Pr[S * S];
#pragma unroll
          for (int i = 0; i < S * S; ++i) Pr[i] = tab(P_s, c, i);
#pragma unroll
          for (int q = 0; q < NS; ++q) {
            double L[S];
            if (code == OP_MSG_ONES) {
#pragma unroll
              for (int s = 0; s < S; ++s) L[s] = live[q] ? 1.0 : 0.0;
            } else if (OBS == OBS_MASK) {
              const unsigned long long mk = live[q]
                  ? reinterpret_cast<const unsigned long long*>(obs)[off_s[ip] + site0 + q * kWalkBlock] : 0ull;
#pragma unroll
              for (int s = 0; s < S; ++s) L[s] = ((mk >> (s ^ fy)) & 1ull) ? 1.0 : 0.0;
            } else {
              const double* d = reinterpret_cast<const double*>(obs) + off_s[ip] + site0 + q * kWalkBlock;
#pragma unroll
              for (int s = 0; s < S; ++s) L[s] = live[q] ? d[(int64_t)(s ^ fy) * stride] : 0.0;
            }
            double G[S];
#pragma unroll
            for (int a = 0; a < S; ++a) {
              double m = 0.0;
#pragma unroll
              for (int b = 0; b < S; ++b) m = fma(Pr[a * S + b], L[b], m);
              G[a] = (RT_WALK_DCHECK(cur[q][a]) m > 0.0) ? cur[q][a] * fast_rcp(m) : 0.0;
            }
#pragma unroll
            for (int i = 0; i < S * S; ++i) w[i] = fma(G[i / S], L[i % S], w[i]);
            if (BR) {
              double x = 0.0;
#pragma unroll
              for (int a = 0; a < S; ++a) {
                double kl = 0.0;
#pragma unroll
                for (int b = 0; b < S; ++b) kl = fma(K_s[c * S * S + a * S + b], L[b], kl);
                x = fma(G[a], kl, x);
              }
              if (site0 + q * kWalkBlock < n_sites) branch_out[(int64_t)c * stride + site0 + q * kWalkBlock] = x;
            }
          }
        }
        // W_c += sum over the warp's 32*NS sites of G (x) L
        reduce_scatter_warp<V, kFramed>(w, lane);
        if (V == 16) {
          if ((lane & 1) == 0 && (lane >> 1) < S * S && w[0] != 0.0)
            atomicAdd(&W_s[c * S * S + (lane >> 1)], w[0]);
        } else if (V == 32) {
          if (lane < S * S && w[0] != 0.0) atomicAdd(&W_s[c * S * S + lane], w[0]);
        } else {
          if (2 * lane < S * S && w[0] != 0.0) atomicAdd(&W_s[c * S * S + 2 * lane], w[0]);
          if (2 * lane + 1 < S * S && w[1] != 0.0) atomicAdd(&W_s[c * S * S + 2 * lane + 1], w[1]);
        }
      }
    };
    double LA[NS][S], LB[NS][S];
    int kA[NS], kB[NS];
#pragma unroll
    for (int q = 0; q < NS; ++q) {
      kA[q] = 0; kB[q] = 0;
#pragma unroll
      for (int s = 0; s < S; ++s) { LA[q][s] = 0.0; LB[q][s] = 0.0; }
    }
    int ip = n_ops - 1;
    issue(ip, LA, kA);
    for (; ip >= 1; ip -= 2) {
      issue(ip - 1, LB, kB);
      do_op(ip, LA, kA);
      issue(ip - 2, LA, kA);
      do_op(ip - 1, LB, kB);
    }
    if (ip == 0) do_op(0, LA, kA);
  }
  __syncthreads();
  for (int i = tid; i < n_nodes * S * S; i += kWalkBlock) {
    const double v = W_s[i];
    if (v != 0.0 && P_s[i] > 0.0) atomicAdd(&W[i], v);
  }
  if (root_post_sum) {
    int t = tid;
    if constexpr (kFramed) asm volatile("mov.u32 %0, %%tid.x;" : "=r"(t));
    if (t < S && rp_s[t] != 0.0) atomicAdd(&root_post_sum[t], rp_s[t]);
  }
}

template <int S, int OBS, bool BR, bool PACKED, bool WEIGHTED>
int launch_walk(int64_t n_sites, int64_t stride, const int4* program, int n_ops, int n_slots,
                int n_nodes, const double* P, const double* root_distn, const void* obs,
                const double* partials, const int8_t* status, double* node_distn, double* W,
                double* root_post_sum, const double* Kmat, double* branch_out,
                const double* site_weight, cudaStream_t stream, bool* handled) {
  constexpr int NS = WalkNS<S>::value;
  auto kern = down_walk_kernel<S, OBS, BR, PACKED, WEIGHTED>;
  const size_t smem = (sizeof(int4) + sizeof(long long)) * n_ops +
                      sizeof(double) * (2 * S + (size_t)n_nodes * ((BR ? 3 : 2) * S * S + S * (S + 1))) +
                      sizeof(double) * (size_t)n_slots * NS * S * kWalkBlock;
  *handled = false;
  if (smem > 100 * 1024) return RT_OK;        // fall back to the level-synchronous kernel
  RT_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 1;
  RT_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kWalkBlock, smem));
  if (per_sm < 1) per_sm = 1;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int64_t tiles = (n_sites + kWalkBlock * NS - 1) / (kWalkBlock * NS);
  int64_t grid = (int64_t)sms * per_sm;
  if (grid > tiles) grid = tiles;
  kern<<<(unsigned)grid, kWalkBlock, smem, stream>>>(n_sites, stride, program, n_ops, n_slots,
                                                     n_nodes, P, root_distn, obs, partials, status,
                                                     node_distn, W, root_post_sum, Kmat, branch_out,
                                                     site_weight);
  RT_CUDA_CHECK(cudaGetLastError());
  *handled = true;
  return RT_OK;
}

// site_weight (nullable): weighted root marginals (see down_walk_kernel); not combined with
// per-branch output
template <int S>
int run(int obs_kind, int64_t n_sites, int64_t stride, const int32_t* program, int n_ops,
        int n_slots, int n_nodes, const int32_t* edges_dev,
        const int32_t* level_ptr_h, int n_levels, const double* P, const double* root_distn,
        const void* obs, const double* partials, const int8_t* status, double* node_distn,
        double* W, double* root_post_sum, const double* Kmat, double* branch_out,
        const double* site_weight, cudaStream_t stream) {
  if (site_weight && branch_out) return RT_ERR_ARG;
  if (program && n_ops > 0) {
    bool handled = false;
    const int4* prog = reinterpret_cast<const int4*>(program);
    int rc = RT_ERR_ARG;
#define RT_WALK(OBSK, PACKED)                                                                     \
  rc = branch_out    ? launch_walk<S, OBSK, true, PACKED, false>(                                  \
                           n_sites, stride, prog, n_ops, n_slots, n_nodes, P, root_distn, obs,      \
                           partials, status, node_distn, W, root_post_sum, Kmat, branch_out,        \
                           nullptr, stream, &handled)                                               \
       : site_weight ? launch_walk<S, OBSK, false, PACKED, true>(                                  \
                           n_sites, stride, prog, n_ops, n_slots, n_nodes, P, root_distn, obs,      \
                           partials, status, node_distn, W, root_post_sum, nullptr, nullptr,        \
                           site_weight, stream, &handled)                                           \
                     : launch_walk<S, OBSK, false, PACKED, false>(                                 \
                           n_sites, stride, prog, n_ops, n_slots, n_nodes, P, root_distn, obs,      \
                           partials, status, node_distn, W, root_post_sum, nullptr, nullptr,        \
                           nullptr, stream, &handled)
    if (obs_kind == OBS_CODES) RT_WALK(OBS_CODES, false);
    else if (obs_kind == 3) RT_WALK(OBS_CODES, true);
    else if (obs_kind == OBS_MASK) RT_WALK(OBS_MASK, false);
    else if (obs_kind == OBS_DENSE) RT_WALK(OBS_DENSE, false);
#undef RT_WALK
    if (rc != RT_OK || handled) return rc;
  }
  // Level-synchronous kernels: the walk's per-node tables do not fit in shared memory.  They pass
  // node marginals through global memory; without a caller's buffer the sites go in chunks through
  // a workspace of kFallbackChunk sites.
  if (obs_kind < 0 || obs_kind > 3) return RT_ERR_ARG;
  constexpr int64_t kFallbackChunk = 1 << 16;
  double* ws = nullptr;
  if (!node_distn) {
    // rows = store indices: one per internal node.  The upward program has one message per edge
    // (n_nodes - 1) and, per internal node, one OP_STORE / OP_ROOT and at most one OP_APPLY_OBS,
    // so n_ops - (n_nodes - 1) is at least the number of internal nodes and at most twice it
    int64_t rows = (int64_t)n_ops - (n_nodes - 1);
    if (rows < 1) rows = 1;
    if (rows > n_nodes) rows = n_nodes;
    const int64_t cs = n_sites < kFallbackChunk ? n_sites : kFallbackChunk;
    RT_CUDA_CHECK(rt_ws_alloc((void**)&ws, sizeof(double) * (size_t)rows * S * cs, stream));
  }
  const int4* edges = reinterpret_cast<const int4*>(edges_dev);
  const int64_t step = ws ? kFallbackChunk : n_sites;
  for (int64_t lo = 0; lo < n_sites; lo += step) {
    const int64_t n = (n_sites - lo < step) ? n_sites - lo : step;
    // every per-site array is site-minor: chunk `lo` starts at element lo of each row
    // (RT_OBS_CODES4 holds two sites per byte, and chunks start at even sites)
    const void* ob = obs;
    if (obs_kind == OBS_DENSE) ob = reinterpret_cast<const double*>(obs) + lo;
    else if (obs_kind == OBS_MASK) ob = reinterpret_cast<const unsigned long long*>(obs) + lo;
    else if (obs_kind == OBS_CODES) ob = reinterpret_cast<const uint8_t*>(obs) + lo;
    else ob = reinterpret_cast<const uint8_t*>(obs) + lo / 2;
    const int64_t nd_stride = ws ? n : stride;
    double* nd = ws ? ws : node_distn + lo;
    double* br = branch_out ? branch_out + lo : nullptr;
    int64_t gr = (n + kBlock - 1) / kBlock;
    int grid_root = (int)(gr < 148 * 8 ? gr : 148 * 8);
    root_distn_kernel<S><<<grid_root, kBlock, 0, stream>>>(n, stride, nd_stride, root_distn, partials + lo,
                                                           status + lo, site_weight ? site_weight + lo : nullptr,
                                                           nd, root_post_sum);
#define RT_LEVELS(OBSK, PACKED)                                                                     \
  (br ? launch_levels<S, OBSK, true, PACKED>(n, stride, nd_stride, edges, level_ptr_h, n_levels, P, ob, \
                                             partials + lo, status + lo, nd, W, Kmat, br, stream)     \
      : launch_levels<S, OBSK, false, PACKED>(n, stride, nd_stride, edges, level_ptr_h, n_levels, P, ob, \
                                              partials + lo, status + lo, nd, W, nullptr, nullptr, stream))
    if (obs_kind == OBS_CODES) RT_LEVELS(OBS_CODES, false);
    else if (obs_kind == 3) RT_LEVELS(OBS_CODES, true);
    else if (obs_kind == OBS_MASK) RT_LEVELS(OBS_MASK, false);
    else RT_LEVELS(OBS_DENSE, false);
#undef RT_LEVELS
  }
  if (ws) RT_CUDA_CHECK(rt_ws_free(ws, stream));
  RT_CUDA_CHECK(cudaGetLastError());
  return RT_OK;
}

}  // namespace

int rt_posterior_small_dispatch(int S, int obs_kind, int64_t n_sites, int64_t stride,
                                const int32_t* program, int n_ops, int n_slots, int n_nodes,
                                const int32_t* edges_dev, const int32_t* level_ptr_h, int n_levels,
                                const double* P, const double* root_distn, const void* obs,
                                const double* partials, const int8_t* status, double* node_distn,
                                double* W, double* root_post_sum, const double* Kmat,
                                double* branch_out, const double* site_weight, cudaStream_t stream) {
#define RT_ARGS obs_kind, n_sites, stride, program, n_ops, n_slots, n_nodes, edges_dev, level_ptr_h, \
                n_levels, P, root_distn, obs, partials, status, node_distn, W, root_post_sum, Kmat,  \
                branch_out, site_weight, stream
  switch (S) {
    case 2: return run<2>(RT_ARGS);
    case 3: return run<3>(RT_ARGS);
    case 4: return run<4>(RT_ARGS);
    case 5: return run<5>(RT_ARGS);
    case 6: return run<6>(RT_ARGS);
    case 7: return run<7>(RT_ARGS);
    case 8: return run<8>(RT_ARGS);
  }
#undef RT_ARGS
  return RT_ERR_UNSUPPORTED;
}
