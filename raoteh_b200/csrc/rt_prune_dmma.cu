// K3: Felsenstein pruning for large state spaces (9 <= S <= 64, e.g. 61 codons)
// on the FP64 tensor pipe (mma.sync m8n8k4 f64 -> SASS DMMA.8x8x4).
//
// Replaces, batched over sites, pyfelscore.mcy_esd_get_node_to_pmap
// (raoteh/sampler/_mcy_dense.py:286-291, spec _mcy.py:611-682, emissions
// _mcz.py:138-163) + _mc0_dense.get_likelihood (_mc0_dense.py:147-212).
//
// One persistent CTA per SM; a tile is 128 sites and every warp walks the whole upward program
// for its own site columns, INDEPENDENTLY of the other warps: there is no block barrier inside
// the walk.  A message is the dense contraction
//     M^T[s, site] = sum_s' P_c[s, s'] * L_c^T[s', site]
// i.e. A = P_c (states x states), B = L_c^T (states x sites), C = messages.
// A warp's B operand is always its own earlier output: warps share only P_c, which goes
// through a ring of three shared-memory buffers filled by TMA bulk copies (cp.async.bulk +
// mbarrier "full"); a warp that is done with a buffer bumps the buffer's counter and the LAST
// of the warps to do so re-arms the barrier and issues the copy of the edge three ahead, so
// nobody ever blocks as a producer and warps may drift up to two edges apart.
// The FP64 tensor pipe belongs to an SM sub-partition, which hosts four of the 16 warps; they
// run free, so one warp's bookkeeping (product over children, mask, exact power-of-two rescale,
// stores, leaf gathers) runs under another warp's DMMAs.  (Round 1 ran two 4-warp CTAs per SM in
// lockstep, with a block barrier per edge and a one-time nanosleep offset between the CTAs;
// making the warps of a sub-partition take turns on the pipe was measured slower,
// profiles/r2_prune_dmma_variants.md.)
// The product over children, the observation mask, the rescale and the root combine run on the C
// fragments in registers; a finished partial goes to the warp's private shared tile (the next B
// operand) and, coalesced, to HBM.  A leaf message with a hard code is one column of P_c per
// site, gathered from a transposed copy of P_c in L2 (no flops, no staging); the tile's leaf
// codes are staged in shared memory at the top of the tile.
// P_c is stored XOR-swizzled (column ^ 4*(row&3)) so fragment loads are bank-conflict
// free without padding.
#include "rt_common.cuh"

namespace {

// One n-tile (8 sites) per warp: 16 warps x 8 sites, <= 128 registers, four warps per SM
// sub-partition to cover the latency-bound bookkeeping between the DMMA phases, at 1.125 shared-
// memory fragment loads per DMMA.  (8 warps x 16 sites, ~250 registers, 0.625 loads per DMMA was
// measured slower at C3 size, profiles/r2_prune_dmma_variants.md.)
constexpr int kNT = 1;                        // n-tiles per warp
constexpr int kWarps = 16;
constexpr int kThreads = 32 * kWarps;
constexpr int kWarpSites = 8 * kNT;
constexpr int kLdB = kWarpSites + 4;          // B tile row stride (== 4 mod 8 -> conflict-free)
constexpr int kFillRows = 32 / kWarpSites;    // rows of the B tile one warp fills per step
#ifndef RT_PD_PROFILE
#define RT_PD_PROFILE 0
#endif
#if RT_PD_PROFILE
// per-phase cycle counters of the pruning kernel (debug builds only: -DRT_PD_PROFILE=1), summed
// over warps: 0 tile loop, 1 leaf gathers, 2 B-tile fills, 3 wait for P_c, 4 unused, 5 DMMA
// loop, 6 release + product, 7 store / root, 8 code staging, 9 other ops
__device__ unsigned long long g_pd_prof[16];
#define RT_PROF_DECL long long prof_t0 = 0, prof_acc[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
#define RT_PROF_BEGIN prof_t0 = clock64();
#define RT_PROF_END(k) prof_acc[k] += clock64() - prof_t0;
#else
#define RT_PROF_DECL
#define RT_PROF_BEGIN
#define RT_PROF_END(k)
#endif
constexpr int kTileSites = kWarps * kWarpSites;   // sites per CTA tile
constexpr int kMaxSlots = 32;
#ifndef RT_PD_RING
#define RT_PD_RING 3
#endif
#ifndef RT_PD_CODE_KB
#define RT_PD_CODE_KB 24
#endif
// (Tried: two P_c buffers and no staged codes, i.e. <= 164 KB of shared memory and ~90 KB of L1
// for the leaf-edge column gathers -- no gain, profiles/r2_prune_dmma_variants.md.)
constexpr int kRing = RT_PD_RING;          // P_c buffers
constexpr int kMaxCodeBytes = RT_PD_CODE_KB * 1024;   // shared-memory budget of the staged leaf codes (0: L1)

__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE;\n"
      "bra WAIT_LOOP;\n"
      "DONE:\n"
      "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
      ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// ---- packing: P[n][S][S] -> Ppad[n][SP][SP] (swizzled), PT[n][SP][SP] (transposed), rowsum[n][SP] ----
__global__ void pack_kernel(const double* __restrict__ P, int S, int SP, int n_nodes,
                            double* __restrict__ Ppad, double* __restrict__ PT,
                            double* __restrict__ rowsum) {
  const int b = blockIdx.x;
  const double* Pb = P + (size_t)b * S * S;
  for (int idx = threadIdx.x; idx < SP * SP; idx += blockDim.x) {
    const int r = idx / SP, c = idx % SP;
    Ppad[(size_t)b * SP * SP + r * SP + (c ^ (4 * (r & 3)))] = (r < S && c < S) ? Pb[r * S + c] : 0.0;
  }
  for (int idx = threadIdx.x; idx < SP * SP; idx += blockDim.x) {
    const int r = idx / SP, c = idx % SP;   // PT[r][c] = P[c][r]
    PT[(size_t)b * SP * SP + idx] = (r < S && c < S) ? Pb[c * S + r] : 0.0;
  }
  for (int r = threadIdx.x; r < SP; r += blockDim.x) {
    double s = 0.0;
    if (r < S)
      for (int c = 0; c < S; ++c) s += Pb[r * S + c];
    rowsum[(size_t)b * SP + r] = s;
  }
}

// MT = number of 8-row m-tiles (padded states SP = 8*MT)
template <int MT, int OBS, bool STORE>
__global__ void __launch_bounds__(kThreads, 1)
prune_dmma_kernel(int S, int64_t n_sites, int64_t stride, const int4* __restrict__ program,
                  int n_ops, int n_slots, const double* __restrict__ Ppad,
                  const double* __restrict__ PT, const double* __restrict__ rowsum,
                  const double* __restrict__ root_distn, const void* __restrict__ obs,
                  double* __restrict__ slots_ws, double* __restrict__ partials,
                  int32_t* __restrict__ exponents, double* __restrict__ loglik,
                  int8_t* __restrict__ status, double* __restrict__ loglik_sum,
                  int code_capacity) {
  constexpr int SP = 8 * MT;
  constexpr int LDP = SP;       // swizzled, no padding
  constexpr int KS = SP / 4;   // k-steps
  extern __shared__ __align__(128) unsigned char smem_raw[];
  double* Pring = reinterpret_cast<double*>(smem_raw);            // [kRing][SP][LDP]
  double* Ball = Pring + (size_t)kRing * SP * LDP;                // [kWarps][SP][kLdB]
  double* pi_s = Ball + (size_t)kWarps * SP * kLdB;               // [SP]
  int* estk = reinterpret_cast<int*>(pi_s + SP);                  // [kWarps][n_slots][kWarpSites]
  int4* prog_s = reinterpret_cast<int4*>(estk + kWarps * n_slots * kWarpSites);
  int* stg_s = reinterpret_cast<int*>(prog_s + n_ops);            // [<= n_ops] node of the i-th staged op
  uint8_t* codes_s = reinterpret_cast<uint8_t*>(stg_s + ((n_ops + 3) & ~3));   // [kWarps][n_code_rows][kWarpSites]
  __shared__ __align__(8) uint64_t full_bar[kRing];
  __shared__ int done_cnt[kRing];
  __shared__ int counts_s[3];      // staged edges per tile, observation rows to stage, observation rows

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  double* Bw = Ball + (size_t)warp * SP * kLdB;
  int* estk_w = estk + warp * n_slots * kWarpSites;

  // edges whose P_c goes through the TMA ring: every contraction.  A leaf with a hard code needs
  // one COLUMN of P_c per site, gathered straight from the transposed copy in L2
  auto needs_stage = [&](const int4& op) -> bool {
    const int code = op.x & 0xff;
    return code == OP_MSG_SLOT || (code == OP_MSG_OBS && OBS != OBS_CODES);
  };
  for (int i = tid; i < n_ops; i += kThreads) prog_s[i] = program[i];
  for (int i = tid; i < SP; i += kThreads) pi_s[i] = (i < S) ? (root_distn ? root_distn[i] : 1.0) : 0.0;
  if (tid < kRing) done_cnt[tid] = 0;
  if (tid == 0) {
    for (int b = 0; b < kRing; ++b) mbar_init(&full_bar[b], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    int k = 0, rows = 0;
    for (int i = 0; i < n_ops; ++i) {
      const int4 op = program[i];
      const int code = op.x & 0xff;
      if (needs_stage(op)) stg_s[k++] = op.y;
      if ((code == OP_MSG_OBS || code == OP_APPLY_OBS) && op.z + 1 > rows) rows = op.z + 1;
    }
    counts_s[0] = k;
    // the tile's leaf codes are staged in shared memory when they fit, else read from global
    counts_s[1] = (OBS == OBS_CODES && rows * kTileSites <= code_capacity) ? rows : 0;
    counts_s[2] = rows;
  }
  __syncthreads();
  const int n_staged = counts_s[0], n_code_rows = counts_s[1], code_rows_all = counts_s[2];
  uint8_t* codes_w = codes_s + (size_t)warp * n_code_rows * kWarpSites;

  const int64_t tiles = (n_sites + kTileSites - 1) / kTileSites;
  const int64_t my_tiles = (tiles - blockIdx.x + gridDim.x - 1) / gridDim.x;
  const long long total_staged = my_tiles * (long long)n_staged;
  // buffer K % kRing holds the P_c of the K-th staged edge of this CTA (K runs on across tiles)
  auto issue = [&](long long K) {
    const int buf = (int)(K % kRing);
    const int node = stg_s[(int)(K % n_staged)];
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    mbar_expect_tx(&full_bar[buf], (uint32_t)(sizeof(double) * SP * LDP));
    tma_load_1d(Pring + (size_t)buf * SP * LDP, Ppad + (size_t)node * SP * LDP,
                (uint32_t)(sizeof(double) * SP * LDP), &full_bar[buf]);
  };
  if (tid == 0)
    for (long long K = 0; K < kRing && K < total_staged; ++K) issue(K);
  long long consumed = 0;          // per warp: staged edges done
  // done with the buffer of staged edge K: the last of the kWarps warps refills it
  auto release = [&](long long K) {
    __syncwarp();
    if (lane == 0) {
      const int buf = (int)(K % kRing);
      __threadfence_block();
      const int old = atomicAdd(&done_cnt[buf], 1);
      if (old == kWarps - 1) {
        done_cnt[buf] = 0;
        __threadfence_block();
        if (K + kRing < total_staged) issue(K + kRing);
      }
    }
  };

  double my_ll = 0.0;
  RT_PROF_DECL
#if RT_PD_PROFILE
  const long long prof_start = clock64();
#endif
  for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    RT_PROF_BEGIN
    // the sites this thread's C-fragment columns map to
    const int64_t site0 = tile * kTileSites + warp * kWarpSites;
    int64_t csite[kNT][2];
    bool cvalid[kNT][2];
#pragma unroll
    for (int j = 0; j < kNT; ++j)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        csite[j][h] = site0 + 8 * j + 2 * t + h;
        cvalid[j][h] = csite[j][h] < n_sites;
      }
    // ---- the warp's leaf codes of this tile: [row][warp sites] bytes in shared memory ----
    if (OBS == OBS_CODES && n_code_rows > 0) {
      __syncwarp();
      const uint8_t* codes = reinterpret_cast<const uint8_t*>(obs);
      const int c = lane % kWarpSites, rh = lane / kWarpSites;
      const bool okc = site0 + c < n_sites;
      for (int r0 = 0; r0 < n_code_rows; r0 += 4 * kFillRows) {   // 4 loads in flight per lane
        uint8_t v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int r = r0 + kFillRows * u + rh;
          v[u] = (r < n_code_rows && okc) ? codes[(int64_t)r * stride + site0 + c] : (uint8_t)RT_MISSING;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int r = r0 + kFillRows * u + rh;
          if (r < n_code_rows) codes_w[r * kWarpSites + c] = v[u];
        }
      }
      __syncwarp();
    }
    if (OBS == OBS_CODES && n_code_rows == 0 && code_rows_all > 0) {
      // codes are read through L1: pull the tile's 128-byte row segments in now
      const uint8_t* codes = reinterpret_cast<const uint8_t*>(obs);
      const int64_t t0 = tile * kTileSites;
      for (int r = tid; r < code_rows_all; r += kThreads)
        if (warp == 0 || true) asm volatile("prefetch.global.L1 [%0];" :: "l"(codes + (int64_t)r * stride + t0));
    }
    RT_PROF_END(8)
    auto code_of = [&](int row, int j, int h) -> int {
      if (n_code_rows > 0) return codes_w[row * kWarpSites + 8 * j + 2 * t + h];
      return cvalid[j][h] ? __ldg(reinterpret_cast<const uint8_t*>(obs) + (int64_t)row * stride + csite[j][h])
                          : RT_MISSING;
    };

    double acc[MT][kNT][2];
    int esum[kNT][2];
#pragma unroll
    for (int i = 0; i < MT; ++i)
#pragma unroll
      for (int j = 0; j < kNT; ++j) acc[i][j][0] = acc[i][j][1] = 1.0;
#pragma unroll
    for (int j = 0; j < kNT; ++j) esum[j][0] = esum[j][1] = 0;
    // `first`: nothing has been multiplied into acc since the last store, so the next message
    // REPLACES it (the FP64 pipe is the DMMA pipe: multiplications by one are skipped)
    bool first = true;

    for (int ip = 0; ip < n_ops; ++ip) {
      const int4 op = prog_s[ip];
      const int code = op.x & 0xff;
      const bool fresh = (op.x >> 8) & 1;

      RT_PROF_BEGIN
      if (code == OP_MSG_OBS && OBS == OBS_CODES) {
        // ---- leaf with hard codes: the message is column k of P_c = row k of PT_c (no flops) ----
        const double* PTc = PT + (size_t)op.y * SP * SP;
        const double* rs = rowsum + (size_t)op.y * SP;
        // branch-free addresses (codes differ from lane to lane): all 4 * MT loads of the lane are
        // issued back to back, then multiplied in; an invalid code (neither a state nor "missing")
        // zeroes the site afterwards under a warp-uniform test
        double col[kNT][2][MT];
        bool bad = false;
#pragma unroll
        for (int j = 0; j < kNT; ++j)
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int k = code_of(op.z, j, h);
            const bool miss = k == RT_MISSING;
            bad = bad || (!miss && k >= S);
            const double* src = (miss ? rs : PTc + (size_t)(k < SP ? k : 0) * SP) + g;
#pragma unroll
            for (int i = 0; i < MT; ++i) col[j][h][i] = __ldg(src + 8 * i);
          }
        if (first) {
#pragma unroll
          for (int j = 0; j < kNT; ++j)
#pragma unroll
            for (int h = 0; h < 2; ++h)
#pragma unroll
              for (int i = 0; i < MT; ++i) acc[i][j][h] = col[j][h][i];
        } else {
#pragma unroll
          for (int j = 0; j < kNT; ++j)
#pragma unroll
            for (int h = 0; h < 2; ++h)
#pragma unroll
              for (int i = 0; i < MT; ++i) acc[i][j][h] *= col[j][h][i];
        }
        first = false;
        if (__any_sync(0xffffffffu, bad)) {
#pragma unroll
          for (int j = 0; j < kNT; ++j)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const int k = code_of(op.z, j, h);
              if (k != RT_MISSING && k >= S) {
#pragma unroll
                for (int i = 0; i < MT; ++i) acc[i][j][h] = 0.0;
              }
            }
        }
        RT_PROF_END(1)
        continue;
      }
      if (needs_stage(op)) {
        const int buf = (int)(consumed % kRing);
        const uint32_t parity = (uint32_t)((consumed / kRing) & 1);
        const double* Ps = Pring + (size_t)buf * SP * LDP;
        // ---- fill the warp's B tile (L_c^T, [SP][warp sites]) --------------------
        if (code == OP_MSG_SLOT) {
          if (!fresh) {
            const double* src = STORE ? partials + (int64_t)op.w * S * stride
                                      : slots_ws + (int64_t)op.z * S * stride;
            __syncwarp();
            {
              const int c = lane % kWarpSites, rh = lane / kWarpSites;
              const bool okc = site0 + c < n_sites;
              const double* sp = src + (int64_t)rh * stride + site0 + c;
              double* bp = Bw + rh * kLdB + c;
#pragma unroll 8
              for (int r0 = 0; r0 < SP; r0 += kFillRows) {
                const double v = (r0 + rh < S && okc) ? __ldcs(sp) : 0.0;
                *bp = v;
                sp += kFillRows * stride;
                bp += kFillRows * kLdB;
              }
            }
          }
#pragma unroll
          for (int j = 0; j < kNT; ++j)
#pragma unroll
            for (int h = 0; h < 2; ++h) esum[j][h] += estk_w[op.z * kWarpSites + 8 * j + 2 * t + h];
        } else {   // OP_MSG_OBS with mask / dense observations at a leaf
          __syncwarp();
          if (OBS == OBS_MASK) {
            const unsigned long long* mk = reinterpret_cast<const unsigned long long*>(obs);
            const int c = lane % kWarpSites;
            const int64_t sg = site0 + c;
            const unsigned long long m = (sg < n_sites) ? mk[(int64_t)op.z * stride + sg] : ~0ull;
            for (int r0 = 0; r0 < SP; r0 += kFillRows) {
              const int r = r0 + lane / kWarpSites;
              Bw[r * kLdB + c] = (r < S && ((m >> r) & 1ull)) ? 1.0 : 0.0;
            }
          } else {
            const double* d = reinterpret_cast<const double*>(obs) + (int64_t)op.z * S * stride;
            for (int r0 = 0; r0 < SP; r0 += kFillRows) {
              const int r = r0 + lane / kWarpSites, c = lane % kWarpSites;
              const int64_t sg = site0 + c;
              double v = (r < S) ? 1.0 : 0.0;
              if (r < S && sg < n_sites) v = d[(int64_t)r * stride + sg];
              Bw[r * kLdB + c] = v;
            }
          }
        }
        __syncwarp();
        RT_PROF_END(2)
        RT_PROF_BEGIN

        // ---- wait for P_c ----
        mbar_wait(&full_bar[buf], parity);
        RT_PROF_END(3)
        RT_PROF_BEGIN
        double msg[MT][kNT][2];
#pragma unroll
        for (int i = 0; i < MT; ++i)
#pragma unroll
          for (int j = 0; j < kNT; ++j) msg[i][j][0] = msg[i][j][1] = 0.0;
#pragma unroll
        for (int kk = 0; kk < KS; ++kk) {
          double bfrag[kNT];
#pragma unroll
          for (int j = 0; j < kNT; ++j) bfrag[j] = Bw[(4 * kk + t) * kLdB + 8 * j + g];
#pragma unroll
          for (int i = 0; i < MT; ++i) {
            const double a = Ps[(8 * i + g) * LDP + 4 * (kk ^ (g & 3)) + t];
#pragma unroll
            for (int j = 0; j < kNT; ++j) dmma884(msg[i][j][0], msg[i][j][1], a, bfrag[j]);
          }
        }
#if RT_PD_PROFILE
        asm volatile("" :: "d"(msg[0][0][0]), "d"(msg[MT - 1][kNT - 1][1]));
#endif
        RT_PROF_END(5)
        RT_PROF_BEGIN
        release(consumed);
        ++consumed;
        if (first) {
#pragma unroll
          for (int i = 0; i < MT; ++i)
#pragma unroll
            for (int j = 0; j < kNT; ++j) { acc[i][j][0] = msg[i][j][0]; acc[i][j][1] = msg[i][j][1]; }
        } else {
#pragma unroll
          for (int i = 0; i < MT; ++i)
#pragma unroll
            for (int j = 0; j < kNT; ++j) { acc[i][j][0] *= msg[i][j][0]; acc[i][j][1] *= msg[i][j][1]; }
        }
        first = false;
        RT_PROF_END(6)
        continue;
      }

      switch (code) {
        case OP_MSG_ONES: {
          first = false;
          const double* rs = rowsum + (size_t)op.y * SP;
#pragma unroll
          for (int i = 0; i < MT; ++i) {
            const double r = rs[8 * i + g];
#pragma unroll
            for (int j = 0; j < kNT; ++j) { acc[i][j][0] *= r; acc[i][j][1] *= r; }
          }
        } break;
        case OP_APPLY_OBS: {
#pragma unroll
          for (int j = 0; j < kNT; ++j)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              if (!cvalid[j][h]) continue;
              if (OBS == OBS_CODES) {
                const int k = code_of(op.z, j, h);
                if (k != RT_MISSING) {
#pragma unroll
                  for (int i = 0; i < MT; ++i) acc[i][j][h] = (8 * i + g == k) ? acc[i][j][h] : 0.0;
                }
              } else if (OBS == OBS_MASK) {
                const unsigned long long m =
                    reinterpret_cast<const unsigned long long*>(obs)[(int64_t)op.z * stride + csite[j][h]];
#pragma unroll
                for (int i = 0; i < MT; ++i) acc[i][j][h] = ((m >> (8 * i + g)) & 1ull) ? acc[i][j][h] : 0.0;
              } else {
                const double* d = reinterpret_cast<const double*>(obs) + (int64_t)op.z * S * stride;
#pragma unroll
                for (int i = 0; i < MT; ++i) {
                  const int s = 8 * i + g;
                  if (s < S) acc[i][j][h] *= d[(int64_t)s * stride + csite[j][h]];
                }
              }
            }
        } break;
        case OP_STORE:
        case OP_ROOT: {
          // rows >= S are padding (only the last m-tile has any): force them to zero so they
          // never win the max
          if (8 * (MT - 1) + g >= S) {
#pragma unroll
            for (int j = 0; j < kNT; ++j) acc[MT - 1][j][0] = acc[MT - 1][j][1] = 0.0;
          }
#pragma unroll
          for (int j = 0; j < kNT; ++j)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              // exponent of the largest entry of the site's column: the entries are non-negative,
              // so the order of the doubles is the order of their high words (one integer max
              // per entry instead of an IEEE fmax)
              int hmx = __double2hiint(acc[0][j][h]);
#pragma unroll
              for (int i = 1; i < MT; ++i) hmx = max(hmx, __double2hiint(acc[i][j][h]));
              hmx = max(hmx, __shfl_xor_sync(0xffffffffu, hmx, 4));
              hmx = max(hmx, __shfl_xor_sync(0xffffffffu, hmx, 8));
              hmx = max(hmx, __shfl_xor_sync(0xffffffffu, hmx, 16));
              // lazy: the column is rescaled only when its largest entry has dropped below
              // 2^-32 (or grown above 1): a partial loses a few bits per node, so most nodes skip
              // the MT multiplications; scaling by powers of two is exact, so the mantissas --
              // and the log-likelihood -- do not depend on when it happens
              const int e_now = (hmx >> 20) - 1023;
              if (hmx >= 0x00100000 && (e_now < -32 || e_now > 0 || code == OP_ROOT)) {
                const int e = e_now;
                const double sc = rt_pow2_neg(e);
#pragma unroll
                for (int i = 0; i < MT; ++i) acc[i][j][h] *= sc;
                esum[j][h] += e;
              }
            }
          // C-fragment layout -> HBM directly: for a fixed m-tile the 8 g-lanes hit 8 rows,
          // the 4 t-lanes 64 contiguous bytes of each row (whole sectors)
          auto store_global = [&](double* dst) {
#pragma unroll
            for (int i = 0; i < MT; ++i) {
              const int s = 8 * i + g;
              if (s < S) {
                double* row = dst + (int64_t)s * stride;
#pragma unroll
                for (int j = 0; j < kNT; ++j)
#pragma unroll
                  for (int h = 0; h < 2; ++h)
                    if (cvalid[j][h]) row[csite[j][h]] = acc[i][j][h];
              }
            }
          };
          if (code == OP_STORE) {
            const bool keep = (op.x >> 9) & 1, park = (op.x >> 10) & 1;
            if (keep) {          // the parent consumes it next: it becomes the warp's B tile
              __syncwarp();
#pragma unroll
              for (int i = 0; i < MT; ++i)
#pragma unroll
                for (int j = 0; j < kNT; ++j) {
                  double2 v = make_double2(acc[i][j][0], acc[i][j][1]);
                  *reinterpret_cast<double2*>(&Bw[(8 * i + g) * kLdB + 8 * j + 2 * t]) = v;
                }
            }
            if (g == 0) {
#pragma unroll
              for (int j = 0; j < kNT; ++j)
#pragma unroll
                for (int h = 0; h < 2; ++h) estk_w[op.z * kWarpSites + 8 * j + 2 * t + h] = esum[j][h];
            }
            if (STORE) store_global(partials + (int64_t)op.w * S * stride);
            else if (park) store_global(slots_ws + (int64_t)op.z * S * stride);
            if (STORE && exponents && g == 0) {
#pragma unroll
              for (int j = 0; j < kNT; ++j)
#pragma unroll
                for (int h = 0; h < 2; ++h)
                  if (cvalid[j][h]) exponents[(int64_t)op.w * stride + csite[j][h]] = esum[j][h];
            }
            __syncwarp();
#pragma unroll
            for (int i = 0; i < MT; ++i)
#pragma unroll
              for (int j = 0; j < kNT; ++j) acc[i][j][0] = acc[i][j][1] = 1.0;
#pragma unroll
            for (int j = 0; j < kNT; ++j) esum[j][0] = esum[j][1] = 0;
            first = true;
          } else {
            if (STORE) store_global(partials + (int64_t)op.w * S * stride);
#pragma unroll
            for (int j = 0; j < kNT; ++j)
#pragma unroll
              for (int h = 0; h < 2; ++h) {
                double lk = 0.0;
#pragma unroll
                for (int i = 0; i < MT; ++i) lk = fma(pi_s[8 * i + g], acc[i][j][h], lk);
                lk += __shfl_xor_sync(0xffffffffu, lk, 4);
                lk += __shfl_xor_sync(0xffffffffu, lk, 8);
                lk += __shfl_xor_sync(0xffffffffu, lk, 16);
                if (g == 0 && cvalid[j][h]) {
                  if (STORE && exponents) exponents[(int64_t)op.w * stride + csite[j][h]] = esum[j][h];
                  if (lk > 0.0) {
                    const double ll = log(lk) + (double)esum[j][h] * RT_LN2;
                    loglik[csite[j][h]] = ll;
                    status[csite[j][h]] = RT_SITE_OK;
                    my_ll += ll;
                  } else {
                    loglik[csite[j][h]] = -INFINITY;
                    status[csite[j][h]] = RT_SITE_STRUCTURAL_ZERO;
                  }
                }
              }
          }
        } break;
        default: break;
      }
      RT_PROF_END((code == OP_STORE || code == OP_ROOT) ? 7 : 9)
    }
  }
#if RT_PD_PROFILE
  if (lane == 0) {
    atomicAdd(&g_pd_prof[0], (unsigned long long)(clock64() - prof_start));
    for (int k = 1; k < 10; ++k) atomicAdd(&g_pd_prof[k], (unsigned long long)prof_acc[k]);
    atomicAdd(&g_pd_prof[10], 1ull);
  }
#endif

  if (loglik_sum) {
    const double w = rt_warp_sum(my_ll);
    if (lane == 0 && w != 0.0) atomicAdd(loglik_sum, w);
  }
}

template <int MT, int OBS, bool STORE>
int launch(int S, int64_t n_sites, int64_t stride, const int4* program, int n_ops, int n_slots,
           const double* Ppad, const double* PT, const double* rowsum, const double* root_distn,
           const void* obs, double* slots_ws, double* partials, int32_t* exponents, double* loglik,
           int8_t* status, double* loglik_sum, cudaStream_t stream) {
  constexpr int SP = 8 * MT;
  constexpr int LDP = SP;
  auto kern = prune_dmma_kernel<MT, OBS, STORE>;
  size_t smem = sizeof(double) * ((size_t)kRing * SP * LDP + (size_t)kWarps * SP * kLdB + SP) +
                sizeof(int) * (size_t)kWarps * n_slots * kWarpSites + sizeof(int4) * (size_t)n_ops +
                sizeof(int) * (((size_t)n_ops + 3) & ~(size_t)3);
  smem = (smem + 15) & ~(size_t)15;
  const size_t limit = 224 * 1024;
  if (smem > limit) return RT_ERR_UNSUPPORTED;
  // whatever is left of the SM's shared memory (one CTA per SM) may hold the tile's leaf codes
  size_t code_capacity = limit - smem;
  if (code_capacity > (size_t)kMaxCodeBytes) code_capacity = kMaxCodeBytes;
  if (OBS != OBS_CODES) code_capacity = 0;
  smem += code_capacity;
  RT_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int64_t tiles = (n_sites + kTileSites - 1) / kTileSites;
  const unsigned grid = (unsigned)(tiles < sms ? tiles : sms);
  kern<<<grid, kThreads, smem, stream>>>(S, n_sites, stride, program, n_ops, n_slots, Ppad, PT,
                                         rowsum, root_distn, obs, slots_ws, partials, exponents,
                                         loglik, status, loglik_sum, (int)code_capacity);
  RT_CUDA_CHECK(cudaGetLastError());
  return RT_OK;
}

template <int MT>
int launch_mt(int S, int obs_kind, bool store, int64_t n_sites, int64_t stride, const int4* program,
              int n_ops, int n_slots, const double* Ppad, const double* PT, const double* rowsum,
              const double* root_distn, const void* obs, double* slots_ws, double* partials,
              int32_t* exponents, double* loglik, int8_t* status, double* loglik_sum,
              cudaStream_t stream) {
#define RT_ARGS S, n_sites, stride, program, n_ops, n_slots, Ppad, PT, rowsum, root_distn, obs, \
                slots_ws, partials, exponents, loglik, status, loglik_sum, stream
#define RT_GO(OBSK) \
  return store ? launch<MT, OBSK, true>(RT_ARGS) : launch<MT, OBSK, false>(RT_ARGS)
  switch (obs_kind) {
    case OBS_CODES: RT_GO(OBS_CODES);
    case OBS_MASK:  RT_GO(OBS_MASK);
    case OBS_DENSE: RT_GO(OBS_DENSE);
  }
#undef RT_GO
#undef RT_ARGS
  return RT_ERR_ARG;
}

}  // namespace

int rt_prune_dmma_dispatch(int S, int obs_kind, bool store, int64_t n_sites, int64_t stride,
                           const int32_t* program, int n_ops, int n_slots, int n_nodes,
                           const double* P, const double* root_distn, const void* obs,
                           double* partials, int32_t* exponents, double* loglik, int8_t* status,
                           double* loglik_sum, cudaStream_t stream) {
  if (n_slots > kMaxSlots) return RT_ERR_UNSUPPORTED;
  const int MT = (S + 15) / 16 * 2;     // padded states 16 / 32 / 48 / 64
  const int SP = 8 * MT, LDP = SP;
  double* ws = nullptr;
  const size_t n_pad = (size_t)n_nodes * SP * LDP, n_rs = (size_t)n_nodes * SP;
  const size_t n_slot = store ? 0 : (size_t)n_slots * S * (size_t)stride;
  RT_CUDA_CHECK(rt_ws_alloc((void**)&ws, sizeof(double) * (2 * n_pad + n_rs + n_slot + 8), stream));
  double* Ppad = ws;
  double* PT = Ppad + n_pad;
  double* rowsum = PT + n_pad;
  double* slots_ws = store ? nullptr : rowsum + n_rs;
  pack_kernel<<<n_nodes, 256, 0, stream>>>(P, S, SP, n_nodes, Ppad, PT, rowsum);
  const int4* prog = reinterpret_cast<const int4*>(program);
  int rc;
#define RT_ARGS S, obs_kind, store, n_sites, stride, prog, n_ops, n_slots, Ppad, PT, rowsum, \
                root_distn, obs, slots_ws, partials, exponents, loglik, status, loglik_sum, stream
  switch (MT) {
    case 2: rc = launch_mt<2>(RT_ARGS); break;
    case 4: rc = launch_mt<4>(RT_ARGS); break;
    case 6: rc = launch_mt<6>(RT_ARGS); break;
    case 8: rc = launch_mt<8>(RT_ARGS); break;
    default: rc = RT_ERR_UNSUPPORTED;
  }
#undef RT_ARGS
  rt_ws_free(ws, stream);
  return rc;
}

#if RT_PD_PROFILE
extern "C" int rt_debug_prune_profile(unsigned long long* out11) {
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(out11, g_pd_prof, sizeof(unsigned long long) * 11);
  unsigned long long z[16] = {0};
  cudaMemcpyToSymbol(g_pd_prof, z, sizeof(z));
  return 0;
}
#endif
