// thrl_scan_lpc.cuh — "lane per chain" scan kernel for the headline shape (2 QTable agents, noise-free demand).
//
// Same game structure as thrl_scan_lut2.cuh (host-built states / compact rows, CTA-built f64 lookup tables), different
// thread mapping.  There a whole warp serves one run, so every instruction of the two sequential dependency chains
// (rollout, update) is issued for 32 lanes but advances one chain; ncu shows that kernel bound by instruction issue and
// shared-memory wavefronts.  Here ONE LANE owns one agent's chain: lanes (2r, 2r+1) are the two agents of run r, a warp
// carries GL/2 runs in its first GL lanes, and every per-chain array is interleaved by lane in shared memory
// (element i of lane l at word i*GL + l  =>  bank == l mod GL: any per-lane index is conflict-free, one wavefront per
// warp instruction).  A row max is GL-wide SIMD over A sequential LDS + FMNMX, the table is lane-private (no warp
// reduction, no fence), and one instruction advances GL chains.  Lane-parallel work (Philox draws) uses all 32 lanes.
//
// Restated reference lines: as in thrl_scan_lut2.cuh / include/thrl.h.
#pragma once
#include "thrl_device.cuh"
#include "thrl_scan_lut2.cuh"

namespace thrl {

__device__ __forceinline__ float lpc_max(float a, float b) { return fmaxf(a, b); }   // FMNMX (values are never NaN)
__device__ __forceinline__ double lpc_max(double a, double b) { return fmax(a, b); }

struct LpcLayout {  // bytes, per warp (all arrays interleaved by lane: [index][GL])
  int off_tab, off_old, off_rec, off_pre, off_gj, off_rows, off_grow, off_eps, off_xrow, warp_bytes;
  int cells_max, rows_max;
};

constexpr int kLpcMaxWarps = 16;

// kA > 0: both agents have exactly kA actions, known at compile time (row loads unrolled, tree max); kA == 0: runtime.
template <typename QT, int GL, int kA>
__global__ void __launch_bounds__(32 * kLpcMaxWarps, 1) qtable_scan_lpc(const __grid_constant__ Lut2Params p, const LpcLayout lay) {
  extern __shared__ __align__(16) unsigned char smem[];
  const ThrlGame& G = p.game;
  const int lane = threadIdx.x & 31, warps_per_cta = blockDim.x >> 5;
  const int warp = __shfl_sync(kFull, (int)(threadIdx.x >> 5), 0);
  const int T = G.max_steps, E = p.E, J = p.J, NS = p.NS;
  const int A0 = kA > 0 ? kA : G.agent[0].actions, A1 = kA > 0 ? kA : G.agent[1].actions;
  const int NR0 = p.NR[0], NR1 = p.NR[1];
  const int rng_mode = p.rng_mode;
  const uint32_t key0 = p.k0, key1 = p.k1;
  constexpr int RPW = GL / 2;  // runs per warp

  // ---------------------------------------------------------------- CTA-shared lookup tables (as in the lut2 kernel)
  uint16_t* nextS = reinterpret_cast<uint16_t*>(smem + p.off_next);       // joint action -> next state
  uint16_t* rowlist = reinterpret_cast<uint16_t*>(smem + p.off_rowlist);  // compact row -> table row, [NR0][NR1]
  double* lutR = reinterpret_cast<double*>(smem + p.off_lutr);            // [J][2] reward (environments.py:34)
  double* lutLog = reinterpret_cast<double*>(smem + p.off_lutlog);        // [J][4] r0/T, r1/T, x0/T, x1/T
  {
    const double ab = __ddiv_rn(G.a, G.b);
    for (int j = threadIdx.x; j < J; j += blockDim.x) {
      const int k0 = j / A1, k1 = j - k0 * A1;
      const double x0 = scale_action(k0, A0, G.agent[0].action_lo, G.agent[0].action_hi);
      const double x1 = scale_action(k1, A1, G.agent[1].action_lo, G.agent[1].action_hi);
      const double aq0 = __dmul_rn(ab, x0), aq1 = __dmul_rn(ab, x1);
      const double Q = __dadd_rn(__dadd_rn(0.0, aq0), aq1);
      const double pn = __dsub_rn(G.a, __dmul_rn(G.b, Q));
      const double price = pn > 0.0 ? pn : (pn != pn ? pn : 0.0);
      const double r0 = __dmul_rn(price, aq0), r1 = __dmul_rn(price, aq1);
      lutR[2 * j] = r0;
      lutR[2 * j + 1] = r1;
      lutLog[4 * j + 0] = __ddiv_rn(r0, (double)T);
      lutLog[4 * j + 1] = __ddiv_rn(r1, (double)T);
      lutLog[4 * j + 2] = __ddiv_rn(x0, (double)T);
      lutLog[4 * j + 3] = __ddiv_rn(x1, (double)T);
      nextS[j] = (uint16_t)p.next_state[j];
    }
    for (int c = threadIdx.x; c < NR0 + NR1; c += blockDim.x)
      rowlist[c] = c < NR0 ? p.row_list[0][c] : p.row_list[1][c - NR0];
  }
  __syncthreads();

  // ---------------------------------------------------------------- this warp's slot
  unsigned char* slot = smem + p.cta_bytes_lpc + (size_t)warp * lay.warp_bytes;
  uint8_t* pre_all = slot + lay.off_pre;                           // [T][GL] forced action or 0xFF
  double* eps_sh = reinterpret_cast<double*>(slot + lay.off_eps);  // [GL] current epsilon of every chain
  int16_t* xrow_sh = reinterpret_cast<int16_t*>(slot + lay.off_xrow);  // [2][GL] table rows held in the two extra slots
  const uint32_t* rec_all = reinterpret_cast<const uint32_t*>(slot + lay.off_rec);
  const uint32_t dp_b = (uint32_t)A1 | (1u << 8);

  const long long total_warps = (long long)gridDim.x * warps_per_cta;
  const long long n_groups = (p.n_runs + RPW - 1) / RPW;
  for (long long grp = (long long)blockIdx.x * warps_per_cta + warp; grp < n_groups; grp += total_warps) {
    // lane l < GL owns chain l = agent (l & 1) of run grp*RPW + l/2.  Lanes without a chain (lane >= GL, or past the last
    // run) shadow chain 0: they execute the same instructions on the same addresses and values, and never store.
    const bool live = lane < GL && grp * RPW + (lane >> 1) < p.n_runs;
    const int l = live ? lane : 0;
    const int ag = l & 1;
    const long long r = grp * RPW + (l >> 1);
    const long long rr = r;
    QT* tab = reinterpret_cast<QT*>(slot + lay.off_tab) + l;               // cell i at tab[i * GL]
    QT* oldv = reinterpret_cast<QT*>(slot + lay.off_old) + l;              // snapshot j at oldv[j * GL]      (agents.py:67)
    uint32_t* rec = reinterpret_cast<uint32_t*>(slot + lay.off_rec) + l;   // step t: own k | joint<<8 | update row of the state before t <<24
    uint32_t* gj = reinterpret_cast<uint32_t*>(slot + lay.off_gj) + l;     // state s: greedy k0 | k1<<8 of the pair
    uint16_t* rows = reinterpret_cast<uint16_t*>(slot + lay.off_rows) + l;  // state s: own compact rows act | upd<<8
    uint8_t* grow = slot + lay.off_grow + l;                               // compact row c: own greedy action
    const int A = kA > 0 ? kA : (ag ? A1 : A0);
    const int NR = ag ? NR1 : NR0;
    const uint16_t* rl = rowlist + (ag ? NR0 : 0);
    const int L = p.L[ag];
    const double* lutR_ag = lutR + ag;
    const double* lutLogR = lutLog + ag;
    const double* lutLogX = lutLog + 2 + ag;
    QT* qg = reinterpret_cast<QT*>(p.q) + rr * G.run_stride + G.agent[ag].table_offset;
    double alpha, gamma, epsend, epsstep;
    if (p.hp) {
      const double* h = p.hp + (rr * 2 + ag) * 4;
      alpha = h[0]; gamma = h[1]; epsend = h[2]; epsstep = h[3];
    } else {
      alpha = G.agent[ag].alpha; gamma = G.agent[ag].gamma; epsend = G.agent[ag].eps_end; epsstep = G.agent[ag].eps_step;
    }
    const double oma = __dsub_rn(1.0, alpha);
    double eps = p.eps[rr * 2 + ag];
    const double price_in = p.price[rr];

    // ---- initial state of the call: rows of the incoming price; extra slots NR, NR+1 hold them if they are not compact rows
    int xrow0 = -1, xrow1 = -1;
    int init_ca, init_cu;
    {
      const int ta = act_row(price_in, (float)G.agent[ag].max_state, (float)G.agent[ag].states);
      const int tu = upd_row(price_in, G.agent[ag].max_state, (double)G.agent[ag].states);
      init_ca = -1; init_cu = -1;
      for (int c = 0; c < NR; ++c) {
        const int row = rl[c];
        if (row == ta) init_ca = c;
        if (row == tu) init_cu = c;
      }
      if (init_ca < 0) { init_ca = NR; xrow0 = ta; }
      if (init_cu < 0) { if (tu == ta) init_cu = init_ca; else { init_cu = NR + 1; xrow1 = tu; } }
    }
    auto table_row = [&](int c) { return c < NR ? (int)rl[c] : (c == NR ? xrow0 : xrow1); };

    // ---- stage this chain's compact rows, greedy action per row, per-state caches
    if (live) {
      for (int c = 0; c < NR + 2; ++c) {
        const int row = table_row(c);
        if (row < 0) continue;
        const QT* src = qg + (size_t)row * G.agent[ag].row_stride;
        QT best = src[0];
        int g = 0;
        tab[(c * A) * GL] = best;
        for (int k = 1; k < A; ++k) {
          const QT v = src[k];
          tab[(c * A + k) * GL] = v;
          if (v > best) { best = v; g = k; }  // first maximal index (agents.py:88)
        }
        grow[c * GL] = (uint8_t)g;
      }
      for (int s = 0; s < NS; ++s) {
        const uint32_t rw = p.state_rows[s];
        rows[s * GL] = (uint16_t)(ag ? (rw >> 16) : (rw & 0xffff));
      }
      rows[NS * GL] = (uint16_t)(init_ca | (init_cu << 8));
    }
    if (live) { eps_sh[l] = eps; xrow_sh[l] = (int16_t)xrow0; xrow_sh[GL + l] = (int16_t)xrow1; }
    __syncwarp();
    {
      // greedy pair per state: own action from the own cache, partner's by shuffle
      for (int s = 0; s <= NS; ++s) {
        const int g = live ? grow[(rows[s * GL] & 0xff) * GL] : 0;
        const int gp = __shfl_xor_sync(kFull, g, 1);
        if (live) gj[s * GL] = ag ? (uint32_t)(gp | (g << 8)) : (uint32_t)(g | (gp << 8));
      }
    }
    __syncwarp();

    int sigma = NS;
    uint32_t last_kk = 0xffffffffu;

    for (int e = 0; e < E; ++e) {
      const uint32_t eabs = (uint32_t)(p.epoch_begin + e);

      // ---- A: draws for the whole episode, all 32 lanes cooperate: one Philox call per (run of this warp, step)
      for (int c = lane; c < RPW * T; c += 32) {
        const int t = c / RPW, rho = c - t * RPW;
        const long long rg = grp * RPW + rho;
        int f0 = 0xFF, f1 = 0xFF;
        if (rg < p.n_runs) {
          const double e0 = eps_sh[2 * rho], e1 = eps_sh[2 * rho + 1];
          const long long sidx = ((rg * E + e) * (long long)T + t) * 2;
          if (rng_mode == THRL_RNG_PHILOX) {
            uint32_t x[4];
            philox4x32_10((uint32_t)(p.run_id0 + rg), eabs, (uint32_t)t, kStreamAct << 16, key0, key1, x);
            if (u32_unit(x[0]) < e0) f0 = (int)__umulhi(x[1], (uint32_t)A0);
            if (u32_unit(x[2]) < e1) f1 = (int)__umulhi(x[3], (uint32_t)A1);
          } else if (rng_mode == THRL_RNG_REPLAY_DRAWS) {
            const double2 u = *reinterpret_cast<const double2*>(p.replay_u + sidx);
            const int2 v = *reinterpret_cast<const int2*>(p.replay_ra + sidx);
            if (u.x < e0) f0 = v.x;
            if (u.y < e1) f1 = v.y;
          } else {
            const int2 v = *reinterpret_cast<const int2*>(p.replay_ra + sidx);
            f0 = v.x; f1 = v.y;
          }
        }
        *reinterpret_cast<uint16_t*>(pre_all + t * GL + 2 * rho) = (uint16_t)((f0 & 0xff) | ((f1 & 0xff) << 8));
      }
      __syncwarp();

      // ---- B: the episode (trainer.py:50-67); every lane walks its run's state, logs its own agent (trainer.py:65-66)
      double acc_r = 0.0, acc_x = 0.0;
      {
        const uint16_t* pp = reinterpret_cast<const uint16_t*>(pre_all + (l & ~1));
        uint32_t kk = 0;
#pragma unroll 2
        for (int t = 0; t < T; ++t) {
          const uint32_t f = pp[t * (GL / 2)];                 // forced pair of this run (0xFF = greedy)
          const uint32_t g = gj[sigma * GL];
          const uint32_t keep = ((f & 0xff) == 0xff ? 0xffu : 0u) | ((f >> 8) == 0xff ? 0xff00u : 0u);
          kk = (g & keep) | (f & ~keep & 0xffffu);             // agents.py:80-89 for both agents
          const uint32_t joint = __dp4a(kk, dp_b, 0u);         // k0 * A1 + k1
          const uint32_t k = ag ? (kk >> 8) : (kk & 0xff);
          if (live) rec[t * GL] = k | (joint << 8) | ((uint32_t)(rows[sigma * GL] >> 8) << 24);
          acc_r = __dadd_rn(acc_r, lutLogR[4 * joint]);
          acc_x = __dadd_rn(acc_x, lutLogX[4 * joint]);
          sigma = nextS[joint];
        }
        last_kk = kk;
      }

      // optional per-step traces (parity runs only)
      if (live && (p.trace_actions || p.trace_rewards || (p.trace_prices && ag == 0))) {
        const double ab = __ddiv_rn(G.a, G.b);
        const long long step0 = (r * E + e) * (long long)T;
        for (int t = 0; t < T; ++t) {
          const uint32_t w = rec[t * GL];
          const int k = w & 0xff, joint = (w >> 8) & 0xffff;
          if (p.trace_actions) p.trace_actions[(step0 + t) * 2 + ag] = k;
          if (p.trace_rewards) p.trace_rewards[(step0 + t) * 2 + ag] = lutR_ag[2 * joint];
          if (p.trace_prices && ag == 0) {
            const int k0 = joint / A1, k1 = joint - k0 * A1;
            const double aq0 = __dmul_rn(ab, scale_action(k0, A0, G.agent[0].action_lo, G.agent[0].action_hi));
            const double aq1 = __dmul_rn(ab, scale_action(k1, A1, G.agent[1].action_lo, G.agent[1].action_hi));
            const double pn = __dsub_rn(G.a, __dmul_rn(G.b, __dadd_rn(__dadd_rn(0.0, aq0), aq1)));
            p.trace_prices[step0 + t] = pn > 0.0 ? pn : (pn != pn ? pn : 0.0);
          }
        }
      }

      // ---- C: snapshot of the old values (agents.py:67) and dirty rows, per chain
      unsigned long long dirty = 0;
      bool dirty_all = false;
      if (live) {
        const uint32_t* rp = rec + (size_t)(T - L) * GL;
        QT* op = oldv;
#pragma unroll 4
        for (int j = 0; j < L; ++j) {
          const uint32_t w = rp[j * GL];
          const int k = w & 0xff, cu = w >> 24;
          op[j * GL] = tab[(cu * A + k) * GL];
          if (cu < 64) dirty |= 1ull << cu; else dirty_all = true;
        }
      }
      // visit counters (agents.py:76): fire-and-forget REDs, all 32 lanes over the (step, chain) pairs of this warp
      if (p.counter) {
        __syncwarp();
        for (int idx = lane; idx < T * GL; idx += 32) {
          const int j = idx / GL, lc = idx - j * GL, agc = lc & 1;
          const long long rc_run = grp * RPW + (lc >> 1);
          if (rc_run < p.n_runs && j >= T - p.L[agc]) {
            const uint32_t w = rec_all[idx];
            const int k = w & 0xff, cu = w >> 24;
            const int Ac = kA > 0 ? kA : (agc ? A1 : A0), NRc = agc ? NR1 : NR0;
            const int row = cu < NRc ? (int)rowlist[(agc ? NR0 : 0) + cu] : (int)xrow_sh[(cu - NRc) * GL + lc];
            atomicAdd(p.counter + rc_run * G.run_stride + G.agent[agc].table_offset + (size_t)row * G.agent[agc].row_stride + k, 1u);
          }
        }
      }

      // ---- D: the sequential pass (agents.py:68-76): lane-private table, no reductions, no fences
      if (live) {
        const uint32_t* rp = rec + (size_t)(T - L) * GL;
        const QT* op = oldv;
        const int cu_final = rows[sigma * GL] >> 8;  // update row of the state after the last step
        uint32_t w = L > 0 ? rp[0] : 0u;
        for (int j = 0; j < L; ++j) {
          const uint32_t wn = (j + 1 < L) ? rp[(j + 1) * GL] : ((uint32_t)cu_final << 24);
          const int k = w & 0xff, joint = (w >> 8) & 0xffff, cu = w >> 24, cn = wn >> 24;
          const QT* row = tab + (size_t)(cn * A) * GL;
          QT m;
          if (kA > 0) {  // all loads first, then a max tree (live table, :71)
            QT v[kA > 0 ? kA : 1];
#pragma unroll
            for (int q = 0; q < kA; ++q) v[q] = row[q * GL];
#pragma unroll
            for (int st = 1; st < kA; st *= 2) {
#pragma unroll
              for (int q = 0; q + st < kA; q += 2 * st) v[q] = lpc_max(v[q], v[q + st]);
            }
            m = v[0];
          } else {
            QT m0 = row[0], m1 = row[GL];
            int kk2 = 2;
#pragma unroll 2
            for (; kk2 + 3 < A; kk2 += 4) {
              m0 = lpc_max(m0, row[kk2 * GL]);
              m1 = lpc_max(m1, row[(kk2 + 1) * GL]);
              m0 = lpc_max(m0, row[(kk2 + 2) * GL]);
              m1 = lpc_max(m1, row[(kk2 + 3) * GL]);
            }
            for (; kk2 < A; ++kk2) m0 = lpc_max(m0, row[kk2 * GL]);
            m = lpc_max(m0, m1);
          }
          const double reward = lutR_ag[2 * joint];
          const double c0 = __dmul_rn(oma, (double)op[j * GL]);
          const double nv = __dadd_rn(c0, __dmul_rn(alpha, __dadd_rn(reward, __dmul_rn(gamma, (double)m))));  // :72-74
          tab[(cu * A + k) * GL] = (QT)nv;                                                                     // :75
          w = wn;
        }
      }

      // ---- E: greedy action of the written rows, greedy pairs per state, epsilon decay, logs / statistics
      if (live) {
        auto refresh_row = [&](int c) {
          const QT* row = tab + (size_t)(c * A) * GL;
          QT best = row[0];
          int g = 0;
          if (kA > 0) {
            QT v[kA > 0 ? kA : 1];
#pragma unroll
            for (int q = 1; q < kA; ++q) v[q] = row[q * GL];
#pragma unroll
            for (int q = 1; q < kA; ++q) if (v[q] > best) { best = v[q]; g = q; }
          } else {
            for (int k = 1; k < A; ++k) { const QT v = row[k * GL]; if (v > best) { best = v; g = k; } }
          }
          grow[c * GL] = (uint8_t)g;
        };
        if (dirty_all) for (int c = 64; c < NR + 2; ++c) refresh_row(c);
        while (dirty) { const int c = __ffsll((long long)dirty) - 1; dirty &= dirty - 1; refresh_row(c); }
      }
      __syncwarp();
      for (int s = 0; s <= NS; ++s) {
        const int g = live ? grow[(rows[s * GL] & 0xff) * GL] : 0;
        const int gp = __shfl_xor_sync(kFull, g, 1);
        if (live) gj[s * GL] = ag ? (uint32_t)(gp | (g << 8)) : (uint32_t)(g | (gp << 8));
      }
      eps = __dadd_rn(epsend, __dmul_rn(__dsub_rn(eps, epsend), epsstep));  // agents.py:78, every epoch
      if (live) eps_sh[l] = eps;
      if (live) {
        if (r < p.n_log_runs) {
          if (p.rewards_log) p.rewards_log[(r * E + e) * 2 + ag] = acc_r;
          if (p.actions_log) p.actions_log[(r * E + e) * 2 + ag] = acc_x;
        }
        if (p.stats) {
          unsigned long long* s4 = reinterpret_cast<unsigned long long*>(p.stats) + ((size_t)e * 2 + ag) * THRL_STATS_K;
          atomicAdd(s4 + 0, (unsigned long long)fx_round(__dmul_rn(acc_r, THRL_STATS_SCALE_SUM)));
          atomicAdd(s4 + 1, (unsigned long long)fx_round(__dmul_rn(__dmul_rn(acc_r, acc_r), THRL_STATS_SCALE_SQ)));
          atomicAdd(s4 + 2, (unsigned long long)fx_round(__dmul_rn(acc_x, THRL_STATS_SCALE_SUM)));
          atomicAdd(s4 + 3, (unsigned long long)fx_round(__dmul_rn(__dmul_rn(acc_x, acc_x), THRL_STATS_SCALE_SQ)));
        }
      }
      __syncwarp();
    }

    // ---- write the chain back: only staged rows can have changed
    if (live) {
      for (int c = 0; c < NR + 2; ++c) {
        const int row = table_row(c);
        if (row < 0) continue;
        QT* dst = qg + (size_t)row * G.agent[ag].row_stride;
        for (int k = 0; k < A; ++k) dst[k] = tab[(c * A + k) * GL];
      }
      p.eps[r * 2 + ag] = eps;
      if (ag == 0 && last_kk != 0xffffffffu) {  // environments.py:36 self.state = price of the last step
        const double ab = __ddiv_rn(G.a, G.b);
        const double aq0 = __dmul_rn(ab, scale_action(last_kk & 0xff, A0, G.agent[0].action_lo, G.agent[0].action_hi));
        const double aq1 = __dmul_rn(ab, scale_action((last_kk >> 8) & 0xff, A1, G.agent[1].action_lo, G.agent[1].action_hi));
        const double pn = __dsub_rn(G.a, __dmul_rn(G.b, __dadd_rn(__dadd_rn(0.0, aq0), aq1)));
        p.price[r] = pn > 0.0 ? pn : (pn != pn ? pn : 0.0);
      }
    }
    __syncwarp();
  }
}

}  // namespace thrl
