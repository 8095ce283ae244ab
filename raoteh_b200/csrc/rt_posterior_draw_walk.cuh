// Body of the K9 draw kernels (rt_posterior_draw.cu), one trajectory per thread, included
// inside posterior_draw_kernel (MIX = false) and posterior_draw_mixture_kernel (MIX = true); the
// kernel defines S, OBS, STATS, TT, MIX, the arguments A and the mixture's X.  The walk is textual
// rather than a device function so that the single-class kernel compiles as a kernel body of its
// own: every mixture-only statement sits under `if constexpr (MIX)`.
//
// MIX: first the site's class c from class_post (Philox substream 2, block 0, word 0; the history's
// words stay those of substream 1), then the walk on class c's P, partials and power table (B is
// read from the table, as it differs per thread), with the statistics reduced per class present
// in the block.
  extern __shared__ __align__(16) unsigned char smem_raw[];
  int4* prog_s = reinterpret_cast<int4*>(smem_raw);
  double* B_s = reinterpret_cast<double*>(prog_s + A.n_ops);          // [S][S]
  double* pi_s = B_s + S * S;                                          // [S]
  double* len_s = pi_s + S;                                            // [n_nodes]
  double* dwell_s = len_s + A.n_nodes;                                 // [S][kBlock]
  uint32_t* trans_s = reinterpret_cast<uint32_t*>(dwell_s + (STATS ? S * kBlock : 0));   // [S*S][kBlock]
  int* par_s = reinterpret_cast<int*>(trans_s + (STATS ? S * S * kBlock : 0));           // [n_nodes]
  // MIX: present_s [8] the classes drawn in the block (bit k), then [kBlock] uint8 each thread's class
  uint32_t* present_s = reinterpret_cast<uint32_t*>(par_s + A.n_nodes);
  __shared__ double red[kBlock / 32][S * S + S];

  const int tid = threadIdx.x;
  double mu = A.ws[0];
  int n_pow = (int)A.ws[1];
  const double* Bt = A.ws + kHeader;
  for (int i = tid; i < A.n_ops; i += kBlock) prog_s[i] = A.program[i];
  if constexpr (!MIX)
    for (int i = tid; i < S * S; i += kBlock) B_s[i] = Bt[S * S + (i % S) * S + i / S];
  if (tid < S) pi_s[tid] = A.root_distn ? A.root_distn[tid] : 1.0;
  for (int i = tid; i < A.n_nodes; i += kBlock) { len_s[i] = A.length[i]; par_s[i] = A.parent[i]; }
  if constexpr (MIX) {
    if (tid < 8) present_s[tid] = 0u;
    reinterpret_cast<uint8_t*>(present_s + 8)[tid] = 0xff;
  }
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
    size_t p_off = 0, l_off = 0;     // MIX: class c's P and partials
    if constexpr (MIX) {
      Philox rc = rng;                // the class: word 0 of (substream 2, block 0)
      rc.block(2u, 0u);
      const int cls = draw_class(X.class_post + site, X.class_post_stride, X.K, rc.out[0]);
      if (cls < 0) {
        fail = RT_SITE_STRUCTURAL_ZERO;
      } else {
        X.site_class[traj] = (uint8_t)cls;
        reinterpret_cast<uint8_t*>(present_s + 8)[tid] = (uint8_t)cls;
        atomicOr(&present_s[cls >> 5], 1u << (cls & 31));
        p_off = (size_t)cls * A.n_nodes * S * S;
        l_off = (size_t)cls * X.partials_class_stride;
        const double* wsc = A.ws + (size_t)cls * table_size<S>();
        mu = wsc[0];
        n_pow = (int)wsc[1];
        Bt = wsc + kHeader;
      }
    }
    // ---- root ~ pi * L_root (store index of the OP_ROOT op); after a failed class draw it reads
    // class 0 and the walk below does not start ----
    {
      const int4 op = prog_s[A.n_ops - 1];
      const double* Lp = at_class<MIX>(A.partials, l_off) + (int64_t)op.w * S * A.site_stride + site;
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
        const double* Lp = at_class<MIX>(A.partials, l_off) + (int64_t)op.w * S * A.site_stride + site;
#pragma unroll
        for (int s = 0; s < S; ++s) L[s] = Lp[(int64_t)s * A.site_stride];
      } else if (code == OP_MSG_OBS) {
        load_obs_vec<S, OBS>(A.obs, op.z, A.obs_stride, site, L);
      } else {
#pragma unroll
        for (int s = 0; s < S; ++s) L[s] = 1.0;
      }
      const double* Prow = at_class<MIX>(A.P, p_off) + ((size_t)c * S + xa) * S;
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
            if constexpr (MIX) {
#pragma unroll
              for (int s = 0; s < S; ++s) { ws[s] = __ldg(Bt + S * S + s * S + x) * __ldg(Bm + s); tw += ws[s]; }
            } else {
#pragma unroll
              for (int s = 0; s < S; ++s) { ws[s] = B_s[x * S + s] * __ldg(Bm + s); tw += ws[s]; }
            }
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

  if constexpr (MIX) {
    if (STATS && A.dwell_sum) {
      // one round per class drawn in the block (present_s is block-uniform after the barrier): the
      // warps sum the statistics of that class's threads, then S + S^2 threads add the block's sums
      const int lane = tid & 31;
      __syncthreads();
      for (int wd = 0; wd < 8; ++wd) {
        for (uint32_t bits = present_s[wd]; bits; bits &= bits - 1) {
          const int k = wd * 32 + __ffs(bits) - 1;
          const bool mine_k = reinterpret_cast<const uint8_t*>(present_s + 8)[tid] == k;
          if (__any_sync(0xffffffffu, mine_k)) {
#pragma unroll
            for (int q = 0; q < S + S * S; ++q) {
              const double mine = !mine_k ? 0.0
                                : q < S ? dwell_s[(q < S ? q : 0) * kBlock + tid]
                                        : (double)trans_s[(q >= S ? q - S : 0) * kBlock + tid];
              const double v = rt_warp_sum(mine);
              if (lane == 0) red[tid >> 5][q] = v;
            }
          } else if (lane == 0) {
            for (int q = 0; q < S + S * S; ++q) red[tid >> 5][q] = 0.0;
          }
          __syncthreads();
          if (tid < S + S * S) {
            double t = 0.0;
            for (int i = 0; i < kBlock / 32; ++i) t += red[i][tid];
            if (t != 0.0)
              atomicAdd(tid < S ? &A.dwell_sum[(size_t)k * S + tid] : &A.trans_sum[(size_t)k * S * S + tid - S], t);
          }
          __syncthreads();
        }
      }
    }
  } else {
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
