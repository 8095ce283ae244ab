// K4/K5 for large state spaces (9 <= S <= 64): downward pass, posterior node
// marginals and per-edge sufficient statistics on the FP64 tensor pipe.
//
// Replaces, batched over sites, pyfelscore.mc0_esd_get_node_to_distn
// (raoteh/sampler/_mc0_dense.py:381, spec :400-489), mc0_esd_get_joint_endpoint_distn
// (_mcy_dense.py:205, spec _mc0_dense.py:217-270) and the `joint_prob/cond_prob`
// accumulation of _mjp_dense.get_expected_history_statistics (:502-510,521-533).
//
// Edge-major, level-synchronous: grid = (site chunks) x (edges of the level).
// A CTA stages P_b once and streams 128-site tiles; per tile three DMMA
// contractions
//     m   = P_b   L_b      (states x sites)      normalisers per parent state
//     D_b = L_b o (P_b^T G),  G = D_a / m        child marginal
//     W_b += G L_b^T       (states x states, K = sites)
// run back to back; W_b (= sum_sites J_b / P_b) stays in registers for the whole
// chunk and is flushed with one masked atomicAdd per entry.  The joint J_b is
// never materialised (7.6 MB per site at S = 61).
//
// Leaf edges with hard codes (half of the edges of a binary tree) do not run on
// the tensor pipe at all: down_leaf_scatter_kernel below sums the parent
// marginals by leaf code, one launch for all of them after the level launches.
#include "rt_common.cuh"

namespace {

constexpr int kWarps = 8;
constexpr int kThreads = kWarps * 32;
constexpr int kNT = 2;
constexpr int kWarpSites = 8 * kNT;               // 16
constexpr int kTileSites = kWarps * kWarpSites;   // 128
constexpr int kLd = kWarpSites + 4;               // 20
constexpr int kTilesPerCta = 8;                   // 1024 sites per CTA

__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// site_weight (nullable): D[root] = w_site * norm(pi o L_root); the level kernels and the leaf
// scatter only propagate the root marginal, so W and every marginal of the site carry the weight.
__global__ void __launch_bounds__(256)
root_distn_generic_kernel(int S, int64_t n_sites, int64_t stride,
                          const double* __restrict__ root_distn,
                          const double* __restrict__ partials, const int8_t* __restrict__ status,
                          const double* __restrict__ site_weight,
                          double* __restrict__ node_distn, double* __restrict__ root_post_sum) {
  extern __shared__ double rsum[];   // [S]
  for (int s = threadIdx.x; s < S; s += blockDim.x) rsum[s] = 0.0;
  __syncthreads();
  // whole warps iterate together (the sums over sites are reduced with shuffles: one shared-memory
  // atomic per warp and state, not one per site -- 256 threads on one CAS loop cost 0.19 ms at C3)
  const int64_t n_round = (n_sites + 31) / 32 * 32;
  for (int64_t site = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; site < n_round;
       site += (int64_t)gridDim.x * blockDim.x) {
    const bool in = site < n_sites;
    const bool ok = in && status[site] == RT_SITE_OK;
    double tot = 0.0;
    for (int s = 0; s < S; ++s)
      tot += in ? partials[(int64_t)s * stride + site] * (root_distn ? root_distn[s] : 1.0) : 0.0;
    const double inv = (ok && tot > 0.0) ? (site_weight ? site_weight[site] : 1.0) / tot : 0.0;
    for (int s = 0; s < S; ++s) {
      const double d = in ? partials[(int64_t)s * stride + site] * (root_distn ? root_distn[s] : 1.0) * inv : 0.0;
      if (in) node_distn[(int64_t)s * stride + site] = d;
      if (root_post_sum) {
        const double t = rt_warp_sum(d);
        if ((threadIdx.x & 31) == 0 && t != 0.0) atomicAdd(&rsum[s], t);
      }
    }
  }
  __syncthreads();
  if (root_post_sum)
    for (int s = threadIdx.x; s < S; s += blockDim.x)
      if (rsum[s] != 0.0) atomicAdd(&root_post_sum[s], rsum[s]);
}

// 1/x to ~1 ulp: hardware seed (rcp.approx.ftz.f64) plus two Newton steps; no slow-path
// branch, so the scheduler can keep loads and DMMAs in flight around it.
__device__ __forceinline__ double fast_rcp(double x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  r = r * fma(-x, r, 2.0);
  r = r * fma(-x, r, 2.0);
  return r;
}

// BR: a fourth contraction kl = K_b L_b and, per site, x = sum_a G_a kl_a: the posterior
// expectation on this branch of the statistic with per-edge kernel K (e.g. expected number of
// synonymous / non-synonymous substitutions, examples/code2x3/extras.py:19-132,
// examples/p53/liwen-branch-expectation.py:176-356).  K_b is staged per tile into the G region,
// which is idle between the W contraction of one tile and the G phase of the next.
//
// Latency hiding (ncu, profiles/r1_ncu_full_summary.json: the first version spent 34 % of its
// warp samples on the scoreboard of the D_a and L_b loads): the D_a values of a tile are loaded
// into registers BEFORE the m contraction and the L_b rows (or code bytes) of the NEXT tile
// before the W contraction, so both global latencies run under 256 DMMAs per warp.
// Leaf edges with hard codes skip the m contraction: P L is a column gather from the staged
// P_b (the row sum for an unobserved site).
template <int MT, int OBS, bool BR>
__global__ void __launch_bounds__(kThreads, 1)
down_dmma_kernel(int S, int64_t n_sites, int64_t stride, const int4* __restrict__ edges,
                 const double* __restrict__ P, const void* __restrict__ obs,
                 const double* __restrict__ partials, const int8_t* __restrict__ status,
                 double* __restrict__ node_distn, double* __restrict__ W,
                 const double* __restrict__ Kmat, double* __restrict__ branch_out, int skip_coded_leaves) {
  constexpr int SP = 8 * MT;
  constexpr int LDP = SP + 4;
  constexpr int KS = SP / 4;
  constexpr int NL = SP / 2;          // L rows per lane in the staging layout
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* Ps = reinterpret_cast<double*>(smem_raw);          // [SP][LDP]
  double* Lall = Ps + SP * LDP;                              // [kWarps][SP][kLd]
  double* Gall = Lall + (size_t)kWarps * SP * kLd;           // [kWarps][SP][kLd]
  double* rs_s = Gall + (size_t)kWarps * SP * kLd;           // [SP] row sums of P_b
  double* krs_s = rs_s + SP;                                 // [SP] row sums of K_b (BR only)

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  const int4 e = edges[blockIdx.y];    // (child node, parent store, child store, child obs slot)
  const int b = e.x;
  // coded leaf: down_leaf_scatter_kernel's edge.  (A run-time flag: as a template parameter the
  // same early exit changed the register allocation of the rest and cost 34 % on internal edges.)
  if (skip_coded_leaves && e.z < 0 && e.w >= 0) return;
  for (int idx = tid; idx < SP * LDP; idx += kThreads) {
    const int r = idx / LDP, c = idx % LDP;
    Ps[idx] = (r < S && c < S) ? P[(size_t)b * S * S + r * S + c] : 0.0;
  }
  double* Lw = Lall + (size_t)warp * SP * kLd;
  double* Gw = Gall + (size_t)warp * SP * kLd;
  const double* Dp = node_distn + (int64_t)e.y * S * stride;
  const double* Lc = e.z >= 0 ? partials + (int64_t)e.z * S * stride : nullptr;
  double* Dc = e.z >= 0 ? node_distn + (int64_t)e.z * S * stride : nullptr;
  // 0: stored partial of an internal child, 1: no observation (ones), 2: leaf observation
  const int kind = Lc ? 0 : (e.w < 0 ? 1 : 2);
  const bool gather = (OBS == OBS_CODES) && kind == 2;

  // W rows [8*warp, 8*warp+8) x all columns, accumulated over the whole chunk
  double Wacc[MT][2];
#pragma unroll
  for (int j = 0; j < MT; ++j) Wacc[j][0] = Wacc[j][1] = 0.0;
  __syncthreads();
  if (tid < SP) {
    double sum = 0.0;
    for (int c = 0; c < S; ++c) sum += Ps[tid * LDP + c];
    rs_s[tid] = sum;
  } else if (BR && tid < 2 * SP) {
    const int r = tid - SP;
    double sum = 0.0;
    if (r < S)
      for (int c = 0; c < S; ++c) sum += Kmat[(size_t)b * S * S + r * S + c];
    krs_s[r] = sum;
  }

  // ---- staging layout of L_b^T: lane owns site column lane & 15, rows r0 + (lane >> 4) ------
  const int sc = lane & 15, rh = lane >> 4;
  double lpre[NL];
  int kpre = -1;
  unsigned long long mpre = 0ull;
  bool live_pre = false;
  auto prefetch = [&](int tile) {
    const int64_t tile0 = ((int64_t)blockIdx.x * kTilesPerCta + tile) * kTileSites;
    const int64_t sg = tile0 + warp * kWarpSites + sc;
    live_pre = tile < kTilesPerCta && sg < n_sites && status[sg] == RT_SITE_OK;
    if (!live_pre) return;
    if (kind == 0) {
      const double* src = Lc + (int64_t)rh * stride + sg;
#pragma unroll
      for (int i = 0; i < NL; ++i) lpre[i] = (2 * i + rh < S) ? __ldcs(src + (int64_t)(2 * i) * stride) : 0.0;
    } else if (kind == 2) {
      if (OBS == OBS_CODES) {
        kpre = reinterpret_cast<const uint8_t*>(obs)[(int64_t)e.w * stride + sg];
      } else if (OBS == OBS_MASK) {
        mpre = reinterpret_cast<const unsigned long long*>(obs)[(int64_t)e.w * stride + sg];
      } else {
        const double* src = reinterpret_cast<const double*>(obs) + ((int64_t)e.w * S + rh) * stride + sg;
#pragma unroll
        for (int i = 0; i < NL; ++i) lpre[i] = (2 * i + rh < S) ? __ldcs(src + (int64_t)(2 * i) * stride) : 0.0;
      }
    }
  };
  prefetch(0);
  __syncthreads();     // rs_s complete

  for (int tile = 0; tile < kTilesPerCta; ++tile) {
    const int64_t tile0 = ((int64_t)blockIdx.x * kTilesPerCta + tile) * kTileSites;
    if (tile0 >= n_sites) break;
    const int64_t site0 = tile0 + warp * kWarpSites;

    if (BR && !gather) {
      // the G region is idle until the G tiles of this tile are written (the previous tile's W
      // phase ended with a block barrier): it holds K_b, padded like P_b, for the fourth contraction
      const double* Kb = Kmat + (size_t)b * S * S;
      for (int idx = tid; idx < SP * LDP; idx += kThreads) {
        const int r = idx / LDP, c = idx % LDP;
        Gall[idx] = (r < S && c < S) ? __ldg(&Kb[r * S + c]) : 0.0;
      }
    }
    // ---- stage the prefetched L_b^T tile of this warp: [SP][16 sites] ----------------------
    const int kcur = live_pre ? kpre : -1;          // code of site column sc (gather edges)
    {
      double* dst = Lw + rh * kLd + sc;
      if (kind == 0 || (kind == 2 && OBS == OBS_DENSE)) {
#pragma unroll
        for (int i = 0; i < NL; ++i) dst[2 * i * kLd] = live_pre ? lpre[i] : 0.0;
      } else if (kind == 1) {
#pragma unroll
        for (int i = 0; i < NL; ++i) dst[2 * i * kLd] = (live_pre && 2 * i + rh < S) ? 1.0 : 0.0;
      } else if (OBS == OBS_CODES) {
#pragma unroll
        for (int i = 0; i < NL; ++i) {
          const int r = 2 * i + rh;
          dst[2 * i * kLd] = (live_pre && r < S && (kcur == RT_MISSING || kcur == r)) ? 1.0 : 0.0;
        }
      } else {
#pragma unroll
        for (int i = 0; i < NL; ++i) {
          const int r = 2 * i + rh;
          dst[2 * i * kLd] = (live_pre && r < S && ((mpre >> r) & 1ull)) ? 1.0 : 0.0;
        }
      }
    }
    // ---- D_a of this tile into registers (C-fragment layout), in flight under the m phase ----
    double dpre[MT][kNT][2];
#pragma unroll
    for (int i = 0; i < MT; ++i)
#pragma unroll
      for (int j = 0; j < kNT; ++j)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int s = 8 * i + g;
          const int64_t sg = site0 + 8 * j + 2 * t + h;
          dpre[i][j][h] = (s < S && sg < n_sites) ? Dp[(int64_t)s * stride + sg] : 0.0;
        }
    __syncwarp();

    double m[MT][kNT][2];
    if (gather) {
      // ---- hard codes at a leaf: m = column k of P_b (row sum when unobserved) --------------
#pragma unroll
      for (int j = 0; j < kNT; ++j)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int k = __shfl_sync(0xffffffffu, kcur, 8 * j + 2 * t + h);
#pragma unroll
          for (int i = 0; i < MT; ++i) {
            const int r = 8 * i + g;
            m[i][j][h] = (k == RT_MISSING) ? rs_s[r] : ((k >= 0 && k < S) ? Ps[r * LDP + k] : 0.0);
          }
        }
    } else {
      // ---- m = P L  (rows = parent states, cols = sites) -----------------------------------
#pragma unroll
      for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int j = 0; j < kNT; ++j) m[i][j][0] = m[i][j][1] = 0.0;
#pragma unroll
      for (int kk = 0; kk < KS; ++kk) {
        double bf[kNT];
#pragma unroll
        for (int j = 0; j < kNT; ++j) bf[j] = Lw[(4 * kk + t) * kLd + 8 * j + g];
#pragma unroll
        for (int i = 0; i < MT; ++i) {
          const double a = Ps[(8 * i + g) * LDP + 4 * kk + t];
#pragma unroll
          for (int j = 0; j < kNT; ++j) dmma884(m[i][j][0], m[i][j][1], a, bf[j]);
        }
      }
    }
    // ---- (BR) kl = K L, same shape as m ------------------------------------------------
    double kl[BR ? MT : 1][kNT][2];
    double xs[kNT][2];
    if (BR && gather) {
      // hard codes at a leaf: K L is column k of K_b (its row sum for an unobserved site)
      const double* Kb = Kmat + (size_t)b * S * S;
#pragma unroll
      for (int j = 0; j < kNT; ++j)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int k = __shfl_sync(0xffffffffu, kcur, 8 * j + 2 * t + h);
#pragma unroll
          for (int i = 0; i < MT; ++i) {
            const int r = 8 * i + g;
            kl[BR ? i : 0][j][h] = (r >= S) ? 0.0
                                   : (k == RT_MISSING) ? krs_s[r]
                                   : ((k >= 0 && k < S) ? __ldg(&Kb[r * S + k]) : 0.0);
          }
          xs[j][h] = 0.0;
        }
    } else if (BR) {
      // K_b was staged into the (idle) G region at the top of the tile; every warp reads all of it
      const double* Ks = Gall;
      __syncthreads();
#pragma unroll
      for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int j = 0; j < kNT; ++j) kl[BR ? i : 0][j][0] = kl[BR ? i : 0][j][1] = 0.0;
#pragma unroll
      for (int kk = 0; kk < KS; ++kk) {
        double bf[kNT];
#pragma unroll
        for (int j = 0; j < kNT; ++j) bf[j] = Lw[(4 * kk + t) * kLd + 8 * j + g];
#pragma unroll
        for (int i = 0; i < MT; ++i) {
          const double a = Ks[(8 * i + g) * LDP + 4 * kk + t];
#pragma unroll
          for (int j = 0; j < kNT; ++j) dmma884(kl[BR ? i : 0][j][0], kl[BR ? i : 0][j][1], a, bf[j]);
        }
      }
#pragma unroll
      for (int j = 0; j < kNT; ++j) xs[j][0] = xs[j][1] = 0.0;
      __syncthreads();      // all warps are done with K_b before the G tiles overwrite it
    }
    // ---- G = D_a / m (0 where D_a == 0), written to the warp's G tile ---------------
#pragma unroll
    for (int i = 0; i < MT; ++i)
#pragma unroll
      for (int j = 0; j < kNT; ++j) {
        double gv[2];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const double d = dpre[i][j][h];
          gv[h] = (d > 0.0 && m[i][j][h] > 0.0) ? d * fast_rcp(m[i][j][h]) : 0.0;
          if (BR) xs[j][h] = fma(gv[h], kl[BR ? i : 0][j][h], xs[j][h]);
        }
        *reinterpret_cast<double2*>(&Gw[(8 * i + g) * kLd + 8 * j + 2 * t]) = make_double2(gv[0], gv[1]);
      }
    if (BR) {
      // sum over the 8 row groups g (lanes with equal t), then lane g == 0 writes its 2 sites
#pragma unroll
      for (int j = 0; j < kNT; ++j)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          double v = xs[j][h];
          v += __shfl_xor_sync(0xffffffffu, v, 4);
          v += __shfl_xor_sync(0xffffffffu, v, 8);
          v += __shfl_xor_sync(0xffffffffu, v, 16);
          const int64_t sg = site0 + 8 * j + 2 * t + h;
          if (g == 0 && sg < n_sites) branch_out[(int64_t)b * stride + sg] = v;
        }
    }
    __syncwarp();

    // ---- D_b = L o (P^T G)  (rows = child states) ------------------------------------
    if (Dc) {
      double d2[MT][kNT][2];
#pragma unroll
      for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int j = 0; j < kNT; ++j) d2[i][j][0] = d2[i][j][1] = 0.0;
#pragma unroll
      for (int kk = 0; kk < KS; ++kk) {
        double bf[kNT];
#pragma unroll
        for (int j = 0; j < kNT; ++j) bf[j] = Gw[(4 * kk + t) * kLd + 8 * j + g];
#pragma unroll
        for (int i = 0; i < MT; ++i) {
          const double a = Ps[(4 * kk + t) * LDP + 8 * i + g];   // P^T[8i+g][4kk+t]
#pragma unroll
          for (int j = 0; j < kNT; ++j) dmma884(d2[i][j][0], d2[i][j][1], a, bf[j]);
        }
      }
#pragma unroll
      for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int j = 0; j < kNT; ++j)
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int s = 8 * i + g;
            const int64_t sg = site0 + 8 * j + 2 * t + h;
            if (s < S && sg < n_sites)
              Dc[(int64_t)s * stride + sg] = d2[i][j][h] * Lw[s * kLd + 8 * j + 2 * t + h];
          }
    }
    __syncthreads();   // every warp's L and G tiles are complete

    // next tile's L rows / codes: in flight under the W contraction
    prefetch(tile + 1);

    // ---- W[8*warp.., :] += G L^T over the 128 sites of the tile ------------------------
    if (warp < MT) {
#pragma unroll 4
      for (int ks = 0; ks < kTileSites / 4; ++ks) {
        const int wt = ks >> 2;            // warp tile owning these 4 sites
        const int col = 4 * (ks & 3) + t;  // site column inside that tile
        const double a = Gall[(size_t)wt * SP * kLd + (8 * warp + g) * kLd + col];
        const double* Lt = Lall + (size_t)wt * SP * kLd;
#pragma unroll
        for (int j = 0; j < MT; ++j) {
          const double bb = Lt[(8 * j + g) * kLd + col];
          dmma884(Wacc[j][0], Wacc[j][1], a, bb);
        }
      }
    }
    __syncthreads();   // tiles may be overwritten
  }

  if (warp < MT) {
#pragma unroll
    for (int j = 0; j < MT; ++j)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int r = 8 * warp + g, c = 8 * j + 2 * t + h;
        const double v = Wacc[j][h];
        if (r < S && c < S && v != 0.0 && Ps[r * LDP + c] > 0.0)
          atomicAdd(&W[(size_t)b * S * S + r * S + c], v);
      }
  }
}

// Leaf edges with hard codes, no DMMA at all.  With a one-hot L_b the three contractions of an
// edge collapse: m = P_b[:, k], G = D_a / P_b[:, k], and W_b = sum_sites G L_b^T only ever touches
// column k of the site -- W_b[:, k] = (sum over the sites with code k of D_a) / P_b[:, k].  So a
// coded leaf edge is a column sum of the parent marginals segmented by the code: 512 B of HBM
// per site and edge, one shared-memory read-modify-write per (state, site).  Run as a dense
// G L^T contraction it was 128 of the 506 contraction units of the C3 downward pass.
//
// One thread per parent state r: row r of the CTA's W tile in shared memory belongs to that
// thread alone, so the scatter needs neither atomics nor barriers; the codes are warp-uniform.
// A lane reads 16 consecutive sites of its row per group (128 contiguous bytes, whole sectors),
// the next group in flight under the scatter of the current one.  Sites whose code is unobserved
// (L_b = ones) go to a per-row register and are spread over the row at the flush; invalid codes and
// failed sites land in the pad column.
constexpr int kLeafThreads = 64;
constexpr int kLeafLd = 67;            // odd: lanes (rows) hit distinct banks for one column; 64 = bin, 65 = unobserved
constexpr int kLeafGroup = 16;
constexpr int kLeafSitesPerCta = 2048;
static_assert(kLeafSitesPerCta % 16 == 0, "K16 needs every CTA's first code byte 16-byte aligned");

template <bool V4, bool K16>
__global__ void __launch_bounds__(kLeafThreads, 6)
down_leaf_scatter_kernel(int S, int64_t n_sites, int64_t stride, const int4* __restrict__ edges,
                         const double* __restrict__ P, const uint8_t* __restrict__ obs,
                         const int8_t* __restrict__ status, const double* __restrict__ node_distn,
                         double* __restrict__ W, int sites_per_cta) {
  const int4 e = edges[blockIdx.y];
  if (e.z >= 0 || e.w < 0) return;     // internal child / unobserved leaf: the DMMA kernel's edge
  extern __shared__ double Ws[];       // [64][kLeafLd]; column 64: bin for skipped sites, 65: unobserved sites
  const int r = threadIdx.x, lane = r & 31;
  const bool act = r < S;
  double* Wr = Ws + r * kLeafLd;
  for (int c = 0; c < kLeafLd; ++c) Wr[c] = 0.0;
  const int64_t c0 = (int64_t)blockIdx.x * sites_per_cta;
  const int64_t c1 = c0 + sites_per_cta < n_sites ? c0 + sites_per_cta : n_sites;
  // lanes past the last state read row 0 into rows of the tile that are never flushed
  const double* Dp = node_distn + ((int64_t)e.y * S + (act ? r : 0)) * stride;
  const uint8_t* code = obs + (int64_t)e.w * stride;

  // Codes of a group.  K16 (rows 16-byte aligned): every lane loads the same 16 code bytes with
  // one vector load and picks its bytes with ALU instructions -- the shuffles that broadcast them
  // otherwise share the MIO queue with the read-modify-writes the kernel waits on (short
  // scoreboard: 6.2 stalls per issue, ncu).  The marginal of a site that failed is exactly zero
  // (root_distn_generic_kernel writes 0, the contraction kernel propagates it), so the vector path
  // does not read the status row.  Ragged last group / unaligned rows: one byte per lane + shuffles.
  struct Codes { uint4 v; int k, st; };
  auto load = [&](double (&dn)[kLeafGroup], Codes& kn, int64_t s0) {
    if (s0 + kLeafGroup <= c1) {
      if (V4) {
        // 32 bytes per lane and instruction: one whole sector
#pragma unroll
        for (int i = 0; i < kLeafGroup; i += 4)
          asm volatile("ld.global.v4.f64 {%0,%1,%2,%3}, [%4];"
                       : "=d"(dn[i]), "=d"(dn[i + 1]), "=d"(dn[i + 2]), "=d"(dn[i + 3]) : "l"(Dp + s0 + i));
      } else {
#pragma unroll
        for (int i = 0; i < kLeafGroup; ++i) dn[i] = __ldg(Dp + s0 + i);
      }
      if (K16) {
        kn.v = __ldg(reinterpret_cast<const uint4*>(code + s0));
        return;
      }
    } else {
#pragma unroll
      for (int i = 0; i < kLeafGroup; ++i) dn[i] = s0 + i < c1 ? __ldg(Dp + s0 + i) : 0.0;
    }
    const int64_t sg = s0 + (lane & (kLeafGroup - 1));
    const bool in = sg < c1;
    // both loads issued together and NOT combined here: the first use of a loaded value blocks
    // the warp, so it belongs to the scatter two groups later
    kn.st = in ? (int)reinterpret_cast<const uint8_t*>(status)[sg] : 1;   // (no sign extension: that is a use)
    kn.k = in ? (int)code[sg] : 254;
  };
  auto scatter = [&](const double (&d)[kLeafGroup], const Codes& ks, bool vec) {
    const int kv = ks.st == RT_SITE_OK ? ks.k : 254;     // failed sites and the tail go to the bin
    const unsigned wv[4] = {ks.v.x, ks.v.y, ks.v.z, ks.v.w};
#pragma unroll
    for (int q = 0; q < kLeafGroup; q += 4) {
      int k[4];
      double w[4], v[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        int kk;
        if (K16 && vec) kk = (int)((wv[q / 4] >> (8 * i)) & 0xffu);
        else kk = __shfl_sync(0xffffffffu, kv, q + i);
        k[i] = kk < S ? kk : (kk == RT_MISSING ? 65 : 64);     // unobserved sites have their own column
        w[i] = Wr[k[i]];
      }
      // four read-modify-writes with their loads issued together.  The codes are warp uniform, so
      // "no column repeats among the four" is a uniform branch: then the four adds are independent;
      // otherwise a repeated column takes the running value instead of the stale load.  The
      // stores stay in program order either way.
      const bool rep = (k[1] == k[0]) | (k[2] == k[0]) | (k[2] == k[1]) |
                       (k[3] == k[0]) | (k[3] == k[1]) | (k[3] == k[2]);
      if (!rep) {
#pragma unroll
        for (int i = 0; i < 4; ++i) v[i] = w[i] + d[q + i];
      } else {
        v[0] = w[0] + d[q];
        v[1] = (k[1] == k[0] ? v[0] : w[1]) + d[q + 1];
        v[2] = (k[2] == k[1] ? v[1] : (k[2] == k[0] ? v[0] : w[2])) + d[q + 2];
        v[3] = (k[3] == k[2] ? v[2] : (k[3] == k[1] ? v[1] : (k[3] == k[0] ? v[0] : w[3]))) + d[q + 3];
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) Wr[k[i]] = v[i];
    }
  };
  // three register buffers in rotation: a group is loaded two scatters before its own.  (The
  // parent marginal of a site that passed is a product of non-negative factors: no clamping.)
  double da[kLeafGroup], db[kLeafGroup], dc[kLeafGroup];
  Codes ka, kb, kc;
  ka.v = make_uint4(0, 0, 0, 0); ka.k = 254; ka.st = 1;
  kb = ka; kc = ka;
  const int64_t G = kLeafGroup;
  if (c0 < c1) load(da, ka, c0);
  if (c0 + G < c1) load(db, kb, c0 + G);
  for (int64_t s0 = c0; s0 < c1; s0 += 3 * G) {
    if (s0 + 2 * G < c1) load(dc, kc, s0 + 2 * G);
    scatter(da, ka, s0 + G <= c1);
    if (s0 + G >= c1) break;
    if (s0 + 3 * G < c1) load(da, ka, s0 + 3 * G);
    scatter(db, kb, s0 + 2 * G <= c1);
    if (s0 + 2 * G >= c1) break;
    if (s0 + 4 * G < c1) load(db, kb, s0 + 4 * G);
    scatter(dc, kc, s0 + 3 * G <= c1);
  }
  if (!act) return;
  const double* Pr = P + ((size_t)e.x * S + r) * S;
  double* Wg = W + ((size_t)e.x * S + r) * S;
  // flush: W_b[r][c] += C[r][c] / P_b[r][c] (+ the unobserved sites' share of the row), the P row
  // loaded eight entries at a time ahead of their use
  const double miss = Wr[65];
  double spread = 0.0;
  if (miss != 0.0) {
    double rs = 0.0;
    for (int c = 0; c < S; ++c) rs += Pr[c];
    spread = rs > 0.0 ? miss / rs : 0.0;
  }
  for (int c0f = 0; c0f < S; c0f += 8) {
    double p[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) p[i] = c0f + i < S ? __ldg(Pr + c0f + i) : 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (p[i] > 0.0) {
        const double val = Wr[c0f + i] / p[i] + spread;
        if (val != 0.0) atomicAdd(&Wg[c0f + i], val);
      }
    }
  }
}

template <int MT>
int run(int S, int obs_kind, int64_t n_sites, int64_t stride, const int32_t* edges_dev,
        const int32_t* level_ptr_h, int n_levels, const double* P, const double* root_distn,
        const void* obs, const double* partials, const int8_t* status, double* node_distn,
        double* W, double* root_post_sum, const double* Kmat, double* branch_out,
        const double* site_weight, cudaStream_t stream) {
  constexpr int SP = 8 * MT;
  constexpr int LDP = SP + 4;
  int64_t gr = (n_sites + 255) / 256;
  root_distn_generic_kernel<<<(int)(gr < 1184 ? gr : 1184), 256, sizeof(double) * S, stream>>>(
      S, n_sites, stride, root_distn, partials, status, site_weight, node_distn, root_post_sum);
  const size_t smem = sizeof(double) * ((size_t)SP * LDP + 2 * (size_t)kWarps * SP * kLd + 2 * SP);
  const int4* edges = reinterpret_cast<const int4*>(edges_dev);
  const unsigned gx = (unsigned)((n_sites + kTilesPerCta * kTileSites - 1) / (kTilesPerCta * kTileSites));
  const bool scatter = obs_kind == OBS_CODES && !branch_out;
#define RT_LAUNCH(OBSK)                                                                           \
  if (branch_out) {                                                                               \
    auto kern = down_dmma_kernel<MT, OBSK, true>;                                                 \
    RT_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    kern<<<grid, kThreads, smem, stream>>>(S, n_sites, stride, edges + e0, P, obs, partials,     \
                                           status, node_distn, W, Kmat, branch_out, 0);           \
  } else {                                                                                        \
    auto kern = down_dmma_kernel<MT, OBSK, false>;                                                \
    RT_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    kern<<<grid, kThreads, smem, stream>>>(S, n_sites, stride, edges + e0, P, obs, partials,     \
                                           status, node_distn, W, nullptr, nullptr, scatter ? 1 : 0); \
  }
  for (int l = 0; l < n_levels; ++l) {
    const int e0 = level_ptr_h[l], e1 = level_ptr_h[l + 1];
    if (e1 <= e0) continue;
    dim3 grid(gx, (unsigned)(e1 - e0));
    switch (obs_kind) {
      case OBS_CODES: RT_LAUNCH(OBS_CODES) break;
      case OBS_MASK: RT_LAUNCH(OBS_MASK) break;
      case OBS_DENSE: RT_LAUNCH(OBS_DENSE) break;
      default: return RT_ERR_ARG;
    }
  }
#undef RT_LAUNCH
  if (scatter && level_ptr_h[n_levels] > 0) {
    // every coded leaf edge of the tree in one launch: its parent's marginal is final by now
    const size_t lsm = sizeof(double) * 64 * kLeafLd;
    const int spc = kLeafSitesPerCta;
    dim3 grid((unsigned)((n_sites + spc - 1) / spc), (unsigned)level_ptr_h[n_levels]);
    const bool v4 = stride % 4 == 0 && (reinterpret_cast<uintptr_t>(node_distn) & 31) == 0;
    const bool k16 = v4 && stride % 16 == 0 && (reinterpret_cast<uintptr_t>(obs) & 15) == 0;
    const uint8_t* codes = reinterpret_cast<const uint8_t*>(obs);
    if (k16)
      down_leaf_scatter_kernel<true, true><<<grid, kLeafThreads, lsm, stream>>>(
          S, n_sites, stride, edges, P, codes, status, node_distn, W, spc);
    else if (v4)
      down_leaf_scatter_kernel<true, false><<<grid, kLeafThreads, lsm, stream>>>(
          S, n_sites, stride, edges, P, codes, status, node_distn, W, spc);
    else
      down_leaf_scatter_kernel<false, false><<<grid, kLeafThreads, lsm, stream>>>(
          S, n_sites, stride, edges, P, codes, status, node_distn, W, spc);
  }
  RT_CUDA_CHECK(cudaGetLastError());
  return RT_OK;
}

}  // namespace

int rt_posterior_dmma_dispatch(int S, int obs_kind, int64_t n_sites, int64_t stride,
                               const int32_t* edges_dev, const int32_t* level_ptr_h, int n_levels,
                               const double* P, const double* root_distn, const void* obs,
                               const double* partials, const int8_t* status, double* node_distn,
                               double* W, double* root_post_sum, const double* Kmat,
                               double* branch_out, const double* site_weight, cudaStream_t stream) {
  const int MT = (S + 15) / 16 * 2;
#define RT_ARGS S, obs_kind, n_sites, stride, edges_dev, level_ptr_h, n_levels, P, root_distn, obs, \
                partials, status, node_distn, W, root_post_sum, Kmat, branch_out, site_weight, stream
  switch (MT) {
    case 2: return run<2>(RT_ARGS);
    case 4: return run<4>(RT_ARGS);
    case 6: return run<6>(RT_ARGS);
    case 8: return run<8>(RT_ARGS);
  }
#undef RT_ARGS
  return RT_ERR_UNSUPPORTED;
}
