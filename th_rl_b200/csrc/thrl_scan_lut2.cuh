// thrl_scan_lut2.cuh — the headline kernel: 2 QTable agents, noise-free demand, tables resident in shared memory.
//
// With noise_prob == 0 the environment step (th_rl/environments.py:25-39) is a pure function of the joint action
// (k0,k1): the next price, both rewards and every encode of that price (agents.py:47-49, f32 for acting, f64 for the
// update) are fixed per joint action.  The host groups joint actions by the encodes of their price into NS "states"
// (41 for the example config) and lists, per agent, the table rows those states can ever address (the *compact rows*);
// only those rows (plus the rows of the call's initial price) are staged in shared memory, which more than doubles the
// number of runs resident per SM.  The f64 lookup values themselves (prices, quantities, reward/T, action/T) are computed by every
// CTA in its prologue with the reference's own formulas.
//
// One warp = one run; per epoch:
//   A  draws      lane-parallel Philox (or replay streams) -> per-step forced actions (epsilon is frozen in an episode;
//                 the exploration test is an integer compare against a per-epoch threshold)
//   B  rollout    sequential, two steps per iteration: state -> greedy pair (cached per state) -> forced override ->
//                 joint action -> next state; log sums on lanes 0-3
//   C  snapshot   lane-parallel: stale old value of every transition of the batch (agents.py:67), visit counters (RED),
//                 dirty-row masks; the state before a step is derived from the action record (no state sequence is kept)
//   D  update     sequential (agents.py:68-76) in chunks of 16 transitions; lane i of a half-warp expands transition i of
//                 its agent and keeps cell address / reward / (1-alpha)*old in registers; both agents' chains interleaved;
//                 row max = 1 LDS + 1 CREDUX.MAX; the owning lane stores
//   E  refresh    greedy cache of the rows that were written (lane = row); epsilon decay; logs / statistics
// Shared memory per run: compact tables + ~1.5 KB of scratch (DESIGN.md 4.1): 24 runs per SM at the C2 shape.
#pragma once
#include "thrl_device.cuh"

namespace thrl {

constexpr int kLut2MaxJoint = 1024;  // A0*A1
constexpr int kLut2MaxStates = 254;  // distinct (encode) states; 255 = the call's initial state at most
constexpr int kLut2MaxRows = 253;    // compact rows per agent (+2 slots for the initial price's rows)

struct Lut2Params {
  ThrlGame game;
  long long n_runs, run_id0;
  int epoch_begin, E, rng_mode;
  uint32_t k0, k1;
  void* q;
  uint32_t* counter;
  double* eps;
  double* price;
  const double* hp;
  const double* replay_u;
  const int32_t* replay_ra;
  double* rewards_log;
  double* actions_log;
  long long n_log_runs;
  long long* stats;
  int32_t* trace_actions;
  double* trace_rewards;
  double* trace_prices;
  // host-built structure of the deterministic game
  int J, NS, NR[2], L[2];             // joint actions, states, compact rows per agent, batch length per agent (0 = never fires)
  uint8_t next_state[kLut2MaxJoint];  // joint action -> state
  uint32_t state_rows[kLut2MaxStates];  // state -> compact rows: act0 | upd0<<8 | act1<<16 | upd1<<24
  uint16_t row_list[2][kLut2MaxRows + 3];  // compact row -> table row
  // shared-memory layout
  int cta_bytes, warp_bytes;
  int cta_bytes_lpc;  // qtable_scan_lpc keeps a [J][2] reward table at off_lutr (this kernel: price per joint action + scaled quantities)
  int off_next, off_rowlist, off_lutlog, off_lutr, off_aq;  // CTA-shared
  int off_tab1, off_grow, off_rows, off_gj, off_seq, off_rec, off_scr, off_old;  // per warp (tables of agent 0 at 0)
  // demand noise (kNoise): steps whose intercept was redrawn this episode, and what they produced
  int noisy;                // 1: the noisy instantiation runs (state / row arrays hold max_steps more entries)
  int off_nt, off_nrec;     // per warp: [T] step index of the k-th noise event; [T] f64 price after that step (the redrawn intercept before it)
  const double* replay_new_a;
};

constexpr int kLut2MaxWarps = 24;  // float tables: 6 warps per scheduler at 80 registers
template <typename QT> struct Lut2Warps { static constexpr int kMax = kLut2MaxWarps; };
template <> struct Lut2Warps<double> { static constexpr int kMax = 16; };  // shared memory caps f64 tables at ~12 runs per SM: leave ptxas 128 registers
constexpr int kLut2NoiseWarps = 16;  // noisy instantiation: every reachable row is staged (~16 KB per run), 13-14 runs fit: 128 registers
constexpr int kLut2Chunk = 16;
// Episodes with at most this many exploration steps are played lane-parallel (phase B).  Each event costs one more lane-
// parallel lift and replay of its 32 steps (~37 warp instructions); past ~12 events that costs more than the step-by-step
// rollout (scripts/lut2_sass_budget.py --events).
constexpr int kLut2MaxEvents = 12;  // transitions expanded per pass of the update (16 lanes per agent)

// Row max / first argmax with the column count known to be <= 32 at compile time (kSmallA): one LDS per lane.
template <typename QT, bool kSmallA>
__device__ __forceinline__ QT lut2_row_max(const QT* row_lane, int A, int lane, bool in) {
  QT m = in ? row_lane[0] : NegInf<QT>::v();
  if (!kSmallA) {
    for (int k = lane + 32; k < A; k += 32) { const QT v = row_lane[k - lane]; m = v > m ? v : m; }
  }
  return warp_max(m);
}
template <typename QT, bool kSmallA>
__device__ __forceinline__ int lut2_row_argmax(const QT* row, int A, int lane, bool in) {
  if (!kSmallA) return row_argmax(row, A, lane);
  const QT v = in ? row[lane] : NegInf<QT>::v();
  const QT wm = warp_max(v);
  return (int)__reduce_min_sync(kFull, (in && v == wm) ? (unsigned)lane : 0xffffffffu);
}

// kNoise: demand noise (environments.py:28-31).  The intercept is redrawn in a few steps of an episode only, so the episode
// is the noise-free rollout between those steps: a noise step computes its price, rewards and the four row encodes in f64 /
// f32 as the reference does and opens an EXTRA state (ids NS+1.. within the episode) whose rows are the encodes themselves --
// the host stages every row the price can reach (0 .. row of a - a * sum(min action)), so a compact row is its table row.
// Snapshot, update and refresh see extra states like any other state; their rewards come from the event records.
template <typename QT, bool kSmallA, bool kNoise = false>
__global__ void __launch_bounds__(kNoise ? 32 * kLut2NoiseWarps : 32 * Lut2Warps<QT>::kMax, 1) qtable_scan_lut2(const __grid_constant__ Lut2Params p) {
  extern __shared__ __align__(16) unsigned char smem[];
  const ThrlGame& G = p.game;
  const int lane = threadIdx.x & 31, warps_per_cta = blockDim.x >> 5;
  const int warp = __shfl_sync(kFull, (int)(threadIdx.x >> 5), 0);  // provably warp-uniform
  const int T = G.max_steps, E = p.E, J = p.J, NS = p.NS;
  const int A0 = G.agent[0].actions, A1 = G.agent[1].actions;
  const int NR0 = p.NR[0], NR1 = p.NR[1];
  const int rng_mode = p.rng_mode;
  const uint32_t key0 = p.k0, key1 = p.k1;

  // ---------------------------------------------------------------- CTA-shared lookup tables
  uint16_t* nextS = reinterpret_cast<uint16_t*>(smem + p.off_next);  // joint action -> 4 * next state (byte offset into GJ)
  uint16_t* rowlist = reinterpret_cast<uint16_t*>(smem + p.off_rowlist);  // compact row -> table row, [NR0][NR1]
  // rewards are price(joint) x quantity(action) (environments.py:34): two small tables instead of a [J][2] one, so that a
  // 24th run fits next to the C2 shape's tables (the product is the same single rounding either way)
  double* lutP = reinterpret_cast<double*>(smem + p.off_lutr);            // [J] price after the joint action
  double* lutAq = reinterpret_cast<double*>(smem + p.off_aq);             // [A0 + A1] a/b * scaled action per agent
  double* lutLog = reinterpret_cast<double*>(smem + p.off_lutlog);        // [J][4] r0/T, r1/T, x0/T, x1/T (trainer.py:65-66)
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
      lutP[j] = price;
      lutLog[4 * j + 0] = __ddiv_rn(r0, (double)T);
      lutLog[4 * j + 1] = __ddiv_rn(r1, (double)T);
      lutLog[4 * j + 2] = __ddiv_rn(x0, (double)T);
      lutLog[4 * j + 3] = __ddiv_rn(x1, (double)T);
      nextS[j] = (uint16_t)(4u * p.next_state[j]);
    }
    for (int k = threadIdx.x; k < A0 + A1; k += blockDim.x) {
      const ThrlAgentSpec& sa = G.agent[k < A0 ? 0 : 1];
      lutAq[k] = __dmul_rn(ab, scale_action(k < A0 ? k : k - A0, sa.actions, sa.action_lo, sa.action_hi));
    }
    for (int c = threadIdx.x; c < NR0 + NR1; c += blockDim.x)
      rowlist[c] = c < NR0 ? p.row_list[0][c] : p.row_list[1][c - NR0];
  }
  __syncthreads();

  // ---------------------------------------------------------------- this warp's slot
  unsigned char* slot = smem + p.cta_bytes + (size_t)warp * p.warp_bytes;
  QT* tab0 = reinterpret_cast<QT*>(slot);
  QT* tab1 = reinterpret_cast<QT*>(slot + p.off_tab1);
  uint8_t* grow = slot + p.off_grow;                                 // greedy action per compact row: [NR0+2][NR1+2]
  uint32_t* rowsW = reinterpret_cast<uint32_t*>(slot + p.off_rows);  // [NS+1] state -> compact rows (entry NS = initial state)
  unsigned char* GJb = slot + p.off_gj;                              // [NS+1] u32: state -> greedy g0 | g1<<8
  uint32_t* GJ = reinterpret_cast<uint32_t*>(GJb);
  uint16_t* rec = reinterpret_cast<uint16_t*>(slot + p.off_rec);     // [T] k0 | k1<<8
  uint8_t* seq = slot + p.off_seq;                                   // kNoise: [T+1] state before step t (rebuilt lane-parallel)
  uint2* pre = reinterpret_cast<uint2*>(slot + p.off_old);           // [T] (keep mask, forced value) byte pairs (phases A-B; olds in C-D)
  // phase D chunk: [kLut2Chunk] uint2 = next-row byte offsets of (agent 0, agent 1) for the transitions being applied.  It
  // shares its bytes with GJ: phases C-D never read GJ, and phase E rebuilds it (GJ[NS+1] is written before it is read)
  unsigned char* chunk = slot + p.off_scr;
  QT* olds = reinterpret_cast<QT*>(slot + p.off_old);                // [T][2] stale old values of the batch (agents.py:67)
  uint8_t* nT = slot + p.off_nt;                                     // kNoise: [T] step of the k-th noise event of the episode
  double* nrec = reinterpret_cast<double*>(slot + p.off_nrec);       // kNoise: [T] price after the k-th noise step (rewards = price x quantity)

  const bool in0 = lane < A0, in1 = lane < A1;
  const bool hi_half = lane >= 16;
  const int L0 = p.L[0], L1 = p.L[1];
  const uint32_t dp_b = (uint32_t)A1 | (1u << 8);  // joint = dp4a(k0 | k1<<8, A1 | 1<<8)
  // lanes >= A re-read the last column: harmless for a max, and no masked load / select in the hot loop
  const uint32_t tab0_off = (uint32_t)(reinterpret_cast<unsigned char*>(tab0) - smem);
  const uint32_t tab1_off = (uint32_t)(reinterpret_cast<unsigned char*>(tab1) - smem);
  const uint32_t tab0_lane_off = tab0_off + (uint32_t)sizeof(QT) * (uint32_t)(kSmallA ? (lane < A0 ? lane : A0 - 1) : lane);
  const uint32_t tab1_lane_off = tab1_off + (uint32_t)sizeof(QT) * (uint32_t)(kSmallA ? (lane < A1 ? lane : A1 - 1) : lane);
  const uint32_t chunk_off = (uint32_t)(chunk - smem);
  const uint32_t smem_base = (uint32_t)__cvta_generic_to_shared(smem);

  const long long total_warps = (long long)gridDim.x * warps_per_cta;
  for (long long r = (long long)blockIdx.x * warps_per_cta + warp; r < p.n_runs; r += total_warps) {
    QT* qg0 = reinterpret_cast<QT*>(p.q) + r * G.run_stride;
    QT* qg1 = qg0 + G.agent[1].table_offset;
    uint32_t* cnt0 = p.counter ? p.counter + r * G.run_stride : nullptr;
    uint32_t* cnt1 = cnt0 ? cnt0 + G.agent[1].table_offset : nullptr;
    const uint32_t gid = (uint32_t)(p.run_id0 + r);
    // the run's hyper-parameters of agent ag: alpha, gamma, eps_end, eps_step (k = 0..3).  They are read where they are used
    // (per half once per run; epsilon decay once per epoch) instead of being held across the epoch loop: ten f64 values
    // would take 20 of the 80 registers that the update and its chunk expansion need.
    auto hparam = [&](int ag, int k) -> double {
      if (p.hp) return __ldg(p.hp + r * 8 + ag * 4 + k);
      const ThrlAgentSpec& s = G.agent[ag];
      return k == 0 ? s.alpha : k == 1 ? s.gamma : k == 2 ? s.eps_end : s.eps_step;
    };
    double alpha_h = hparam(hi_half, 0), gamma_h = hparam(hi_half, 1), oma_h = __dsub_rn(1.0, alpha_h);
    asm volatile("" : "+d"(alpha_h), "+d"(gamma_h), "+d"(oma_h));  // keep the selected values live (no re-selection in the loops)
    double eps0 = p.eps[r * 2], eps1 = p.eps[r * 2 + 1];
    const double price_in = p.price[r];

    // ---- the call's initial state: rows of the incoming price, aliased to a compact row when it is one
    int init_c0, init_c1, init_c2, init_c3;            // act0, upd0, act1, upd1 compact indices
    int xrow00 = -1, xrow01 = -1, xrow10 = -1, xrow11 = -1;  // table rows staged in the two extra slots of each agent
    {
      auto find = [&](const uint16_t* rl, int NRa, int row) -> int {
        int res = -1;
        for (int c0 = 0; c0 < NRa; c0 += 32) {
          const unsigned f = __ballot_sync(kFull, c0 + lane < NRa && rl[c0 + lane] == row);
          if (f) { res = c0 + __ffs(f) - 1; break; }
        }
        return res;
      };
      const int ta0 = act_row(price_in, (float)G.agent[0].max_state, (float)G.agent[0].states);
      const int tu0 = upd_row(price_in, G.agent[0].max_state, (double)G.agent[0].states);
      const int ta1 = act_row(price_in, (float)G.agent[1].max_state, (float)G.agent[1].states);
      const int tu1 = upd_row(price_in, G.agent[1].max_state, (double)G.agent[1].states);
      init_c0 = find(rowlist, NR0, ta0);
      if (init_c0 < 0) { init_c0 = NR0; xrow00 = ta0; }
      init_c1 = find(rowlist, NR0, tu0);
      if (init_c1 < 0) { if (tu0 == ta0) init_c1 = init_c0; else { init_c1 = NR0 + 1; xrow01 = tu0; } }
      init_c2 = find(rowlist + NR0, NR1, ta1);
      if (init_c2 < 0) { init_c2 = NR1; xrow10 = ta1; }
      init_c3 = find(rowlist + NR0, NR1, tu1);
      if (init_c3 < 0) { if (tu1 == ta1) init_c3 = init_c2; else { init_c3 = NR1 + 1; xrow11 = tu1; } }
    }
    auto table_row0 = [&](int c) { return c < NR0 ? (int)rowlist[c] : (c == NR0 ? xrow00 : xrow01); };
    auto table_row1 = [&](int c) { return c < NR1 ? (int)rowlist[NR0 + c] : (c == NR1 ? xrow10 : xrow11); };

    // ---- stage compact rows (plus extra rows) into shared memory, build the caches
    for (int c = 0; c < NR0 + 2; ++c) {
      const int row = table_row0(c);
      if (row >= 0) for (int k = lane; k < A0; k += 32) tab0[c * A0 + k] = qg0[(size_t)row * G.agent[0].row_stride + k];
    }
    for (int c = 0; c < NR1 + 2; ++c) {
      const int row = table_row1(c);
      if (row >= 0) for (int k = lane; k < A1; k += 32) tab1[c * A1 + k] = qg1[(size_t)row * G.agent[1].row_stride + k];
    }
    for (int s = lane; s < NS; s += 32) rowsW[s] = p.state_rows[s];
    if (lane == 0) rowsW[NS] = (uint32_t)init_c0 | ((uint32_t)init_c1 << 8) | ((uint32_t)init_c2 << 16) | ((uint32_t)init_c3 << 24);
    __syncwarp();
    for (int c = 0; c < NR0 + 2; ++c) {
      if (table_row0(c) >= 0) {
        const int g = lut2_row_argmax<QT, kSmallA>(tab0 + c * A0, A0, lane, in0);
        if (lane == 0) grow[c] = (uint8_t)g;
      }
    }
    for (int c = 0; c < NR1 + 2; ++c) {
      if (table_row1(c) >= 0) {
        const int g = lut2_row_argmax<QT, kSmallA>(tab1 + c * A1, A1, lane, in1);
        if (lane == 0) grow[NR0 + 2 + c] = (uint8_t)g;
      }
    }
    __syncwarp();
    for (int s = lane; s <= NS; s += 32) {
      const uint32_t rw = rowsW[s];
      GJ[s] = (uint32_t)grow[rw & 0xff] | ((uint32_t)grow[NR0 + 2 + ((rw >> 16) & 0xff)] << 8);
    }
    __syncwarp();

    uint32_t sig4 = 4u * (uint32_t)NS;  // 4 * current state
    int last_k = -1;                    // k0 | k1<<8 of the most recent step (for the outgoing price)
    double noise_price = -1.0;          // kNoise: price after the latest episode when its last step was a noise step (prices are >= 0)

    for (int e = 0; e < E; ++e) {
      const uint32_t eabs = (uint32_t)(p.epoch_begin + e);
      const long long step0 = (r * E + e) * (long long)T;

      // ---- A: draws (agents.py:81-82), lane-parallel over the steps of the episode.
      //      pre[t] = (keep, forced): action pair = (greedy pair & keep) | forced
      const unsigned long long thr0 = u32_unit_threshold(eps0), thr1 = u32_unit_threshold(eps1);  // u32_unit(x) < eps <=> x < thr
      for (int t = lane; t < T; t += 32) {
        int f0, f1;
        if (rng_mode == THRL_RNG_PHILOX) {
          uint32_t x[4];
          philox4x32_10(gid, eabs, (uint32_t)t, kStreamAct << 16, key0, key1, x);
          f0 = x[0] < thr0 ? (int)__umulhi(x[1], (uint32_t)A0) : -1;
          f1 = x[2] < thr1 ? (int)__umulhi(x[3], (uint32_t)A1) : -1;
        } else if (rng_mode == THRL_RNG_REPLAY_DRAWS) {
          const double2 u = *reinterpret_cast<const double2*>(p.replay_u + (step0 + t) * 2);
          const int2 v = *reinterpret_cast<const int2*>(p.replay_ra + (step0 + t) * 2);
          f0 = u.x < eps0 ? v.x : -1;
          f1 = u.y < eps1 ? v.y : -1;
        } else {
          const int2 v = *reinterpret_cast<const int2*>(p.replay_ra + (step0 + t) * 2);
          f0 = v.x; f1 = v.y;
        }
        pre[t] = make_uint2((f0 < 0 ? 0xffu : 0u) | (f1 < 0 ? 0xff00u : 0u),
                            (uint32_t)(f0 < 0 ? 0 : f0) | ((uint32_t)(f1 < 0 ? 0 : f1) << 8));
      }
      int nK = 0;  // noise events of this episode
      if (kNoise) {
        for (int t0 = 0; t0 < T; t0 += 32) {  // environments.py:28-31, lane = step; the events in step order
          const int t = t0 + lane;
          bool ev = false;
          double na = G.a;
          if (t < T) {
            if (rng_mode == THRL_RNG_PHILOX) {
              uint32_t x[4];
              philox4x32_10(gid, eabs, (uint32_t)t, kStreamEnv << 16, key0, key1, x);
              if (u53(x[0], x[1]) < G.noise_prob) {
                const double lo = __dmul_rn(G.a, 0.7);
                na = __dadd_rn(lo, __dmul_rn(__dsub_rn(G.a, lo), u53(x[2], x[3])));
                ev = true;
              }
            } else if (p.replay_new_a) {
              na = p.replay_new_a[step0 + t];
              ev = __double_as_longlong(na) != __double_as_longlong(G.a);
            }
          }
          const unsigned m = __ballot_sync(kFull, ev);
          if (ev) {
            const int idx = nK + __popc(m & ((1u << lane) - 1u));
            nT[idx] = (uint8_t)t;
            nrec[idx] = na;  // the intercept, until the step replaces it by the price
          }
          nK += __popc(m);
        }
      }
      __syncwarp();

      // ---- B: the episode (trainer.py:50-67).  Lanes 0..3 carry the four log accumulators (trainer.py:65-66).
      const uint32_t sig4_start = sig4;
      double acc = 0.0;
      {
        // shared-window addresses in registers and explicit ld/st.shared: one IMAD / IADD per access
        const uint32_t base = (uint32_t)__cvta_generic_to_shared(smem);
        const uint32_t pre_a = base + (uint32_t)(reinterpret_cast<unsigned char*>(pre) - smem);
        const uint32_t rec_a = base + (uint32_t)(reinterpret_cast<unsigned char*>(rec) - smem);
        const uint32_t gj_a = base + (uint32_t)(GJb - smem);
        const uint32_t log_a = base + (uint32_t)p.off_lutlog + 8u * (uint32_t)(lane & 3);
        uint32_t next_a = base + (uint32_t)p.off_next;
        asm volatile("" : "+r"(next_a));  // keep it in a register
        const uint32_t log_lane = lane < 4 ? 1u : 0u;
        double lg = 0.0;
        uint32_t kk = 0;
        // one step: greedy pair of the state, forced override, joint action, log accumulate (lanes 0-3 only), next state
        auto step = [&](uint32_t fx, uint32_t fy) {
          uint32_t gj, s16;
          asm volatile("ld.shared.u32 %0, [%1];" : "=r"(gj) : "r"(gj_a + sig4));
          kk = (gj & fx) | fy;                                 // agents.py:80-89 for both agents
          const uint32_t joint = __dp4a(kk, dp_b, 0u);         // k0 * A1 + k1
          asm volatile("{ .reg .pred q; setp.ne.u32 q, %2, 0; @q ld.shared.f64 %0, [%1]; }"
                       : "+d"(lg) : "r"(log_a + 32u * joint), "r"(log_lane));  // lanes 0-3 only (other lanes keep lg = 0)
          acc = __dadd_rn(acc, lg);                            // trainer.py:65-66
          asm volatile("ld.shared.u16 %0, [%1];" : "=r"(s16) : "r"(next_a + 2u * joint));
          sig4 = s16;
        };
        // Events: steps where an agent explores (keep != 0xffff).  Between events the greedy pairs GJ are frozen, so the next
        // state is a fixed function of the current one, F(s) = nextS[joint(GJ[s])].  With few events the episode is played
        // lane-parallel from the powers of F; otherwise (and past the limits of the lane-parallel plan) step by step.
        unsigned evm0 = 0, evm1 = 0, evm2 = 0, evm3 = 0;  // event masks of steps 0-31, 32-63, 64-95, 96-127
        bool par = false;
        if (!kNoise && T > 0 && T <= 128 && NS < 64) {
          const uint32_t* prew = reinterpret_cast<const uint32_t*>(pre);
          auto evmask = [&](int t0) { const int t = t0 + lane; return __ballot_sync(kFull, t < T && prew[2 * t] != 0xffffu); };
          evm0 = evmask(0); evm1 = evmask(32); evm2 = evmask(64); evm3 = evmask(96);
          par = __popc(evm0) + __popc(evm1) + __popc(evm2) + __popc(evm3) <= kLut2MaxEvents;
        }
        if (!kNoise && par) {
          // ---- B.map: successor powers.  Byte 0 of fp[k] in lane l is F^(2^k)(l), byte 1 is F^(2^k)(l + 32); states past NS
          //      map to themselves.  The rollout goes 32 steps at a time, so five levels cover every distance.
          uint32_t fp[5];
          {
            auto succ = [&](uint32_t s) -> uint32_t {
              uint32_t n4 = 4u * s;
              if (s <= (uint32_t)NS) {
                uint32_t gj;
                asm volatile("ld.shared.u32 %0, [%1];" : "=r"(gj) : "r"(gj_a + 4u * s));
                asm volatile("ld.shared.u16 %0, [%1];" : "=r"(n4) : "r"(next_a + 2u * __dp4a(gj, dp_b, 0u)));
              }
              return n4 >> 2;
            };
            fp[0] = succ((uint32_t)lane) | (succ((uint32_t)lane + 32u) << 8);
          }
          // F^(2^k)(s) from level k's table: lane s & 31 holds it in byte s >> 5 (s < 64: one PRMT, selector 0x4440 + byte)
          auto fwd = [&](uint32_t v, uint32_t s) -> uint32_t {
            uint32_t r;
            asm("prmt.b32 %0, %1, 0, %2;" : "=r"(r) : "r"(__shfl_sync(kFull, v, (int)s)), "r"((s >> 5) + 0x4440u));
            return r;
          };
#pragma unroll
          for (int k = 1; k < 5; ++k) fp[k] = fwd(fp[k - 1], fp[k - 1] & 0xffu) | (fwd(fp[k - 1], fp[k - 1] >> 8) << 8);
          // F^d(s) for d < 32, d per lane
          auto lift = [&](uint32_t s, uint32_t d) -> uint32_t {
#pragma unroll
            for (int k = 0; k < 5; ++k) {
              const uint32_t n = fwd(fp[k], s);
              s = (d >> k) & 1u ? n : s;
            }
            return s;
          };

          uint32_t sc = sig4_start >> 2;  // state before the first step of the 32
          unsigned m = evm0;
          for (int c0 = 0; c0 < T; c0 += 32) {
            // ---- B.fill: lane = step t = c0 + lane.  Its state is F^(t - c0)(sc) up to the first event; each event, in
            //      step order, restarts the lanes after it from the state it leads to.  Every step is played the same way,
            //      events too: action pair = (greedy pair & keep) | forced, and the state it leads to (n4 = 4 x state)
            const int t = c0 + lane;
            uint32_t fx = 0xffffu, fy = 0u;
            if (t < T) asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(fx), "=r"(fy) : "r"(pre_a + 8u * (uint32_t)t));
            uint32_t st = lift(sc, (uint32_t)lane), kt, n4;
            auto play = [&]() {
              uint32_t gj;
              asm volatile("ld.shared.u32 %0, [%1];" : "=r"(gj) : "r"(gj_a + 4u * st));
              kt = (gj & fx) | fy;
              asm volatile("ld.shared.u16 %0, [%1];" : "=r"(n4) : "r"(next_a + 2u * __dp4a(kt, dp_b, 0u)));
            };
            play();
            for (unsigned mw = m; mw != 0u; mw &= mw - 1u) {
              const int i = __ffs(mw) - 1;
              const uint32_t nx = lift(__shfl_sync(kFull, n4, i) >> 2, (uint32_t)(lane - i - 1));
              st = lane > i ? nx : st;
              play();
            }
            if (t < T) asm volatile("st.shared.u16 [%0], %1;" ::"r"(rec_a + 2u * (uint32_t)t), "h"((uint16_t)kt) : "memory");
            sc = __shfl_sync(kFull, n4, 31) >> 2;
            m = c0 == 0 ? evm1 : c0 == 32 ? evm2 : evm3;
          }
          __syncwarp();
          // ---- B.log: the four log sums in step order on lanes 0-3 (trainer.py:65-66), one DADD per step.  The lutLog
          //      address of a step is one DP2A of its action pair: base + 32 A1 k0 + 32 k1
          {
            const uint32_t lq = log_a, wq = (32u * (uint32_t)A1) | (32u << 16);
            auto add = [&](uint32_t a) {
              asm volatile("ld.shared.f64 %0, [%1];" : "=d"(lg) : "r"(a));
              acc = __dadd_rn(acc, lg);
            };
            auto eight = [&](int t) {  // eight steps per 16-byte load of rec
              uint32_t r0, r1, r2, r3;
              asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(rec_a + 2u * (uint32_t)t));
              add(__dp2a_lo(wq, r0, lq)); add(__dp2a_hi(wq, r0, lq));
              add(__dp2a_lo(wq, r1, lq)); add(__dp2a_hi(wq, r1, lq));
              add(__dp2a_lo(wq, r2, lq)); add(__dp2a_hi(wq, r2, lq));
              add(__dp2a_lo(wq, r3, lq)); add(__dp2a_hi(wq, r3, lq));
            };
            int t = 0;
#pragma unroll 1
            for (; t + 32 <= T; t += 32) { eight(t); eight(t + 8); eight(t + 16); eight(t + 24); }
#pragma unroll 1
            for (; t + 8 <= T; t += 8) eight(t);
#pragma unroll 1
            for (; t < T; ++t) {
              uint32_t r0;
              asm volatile("ld.shared.u16 %0, [%1];" : "=r"(r0) : "r"(rec_a + 2u * (uint32_t)t));
              add(__dp2a_lo(wq, r0, lq));
            }
          }
          uint32_t s16;
          asm volatile("ld.shared.u16 %0, [%1];" : "=r"(kk) : "r"(rec_a + 2u * (uint32_t)(T - 1)));
          asm volatile("ld.shared.u16 %0, [%1];" : "=r"(s16) : "r"(next_a + 2u * __dp4a(kk, dp_b, 0u)));
          sig4 = s16;
        } else if (!kNoise) {
        uint32_t pa = pre_a, ra = rec_a;
#pragma unroll 2
        for (int n2 = T >> 1; n2 > 0; --n2, pa += 16u, ra += 4u) {  // two steps per 16-byte load of pre and per 4-byte store of rec
          uint32_t f0x, f0y, f1x, f1y;
          asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(f0x), "=r"(f0y), "=r"(f1x), "=r"(f1y) : "r"(pa));
          step(f0x, f0y);
          const uint32_t ka = kk;
          step(f1x, f1y);
          asm volatile("st.shared.u32 [%0], %1;" ::"r"(ra), "r"(__byte_perm(ka, kk, 0x5410)) : "memory");  // same value from every lane
        }
        if (T & 1) {
          uint32_t fx, fy;
          asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(fx), "=r"(fy) : "r"(pa));
          step(fx, fy);
          asm volatile("st.shared.u16 [%0], %1;" ::"r"(ra), "h"((uint16_t)kk) : "memory");
        }
        } else {
          // the noise-free rollout between the noise steps: single steps up to an even step index, pairs, a single tail step
          auto single = [&](int t) {
            uint32_t fx, fy;
            asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(fx), "=r"(fy) : "r"(pre_a + 8u * (uint32_t)t));
            step(fx, fy);
            asm volatile("st.shared.u16 [%0], %1;" ::"r"(rec_a + 2u * (uint32_t)t), "h"((uint16_t)kk) : "memory");
          };
          const double ab = __ddiv_rn(G.a, G.b), Td = (double)T;
          int t = 0;
          for (int k = 0; k <= nK; ++k) {
            const int tn = k < nK ? (int)nT[k] : T;
            if (t < tn && (t & 1)) { single(t); ++t; }
            for (; t + 1 < tn; t += 2) {
              uint32_t f0x, f0y, f1x, f1y;
              asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(f0x), "=r"(f0y), "=r"(f1x), "=r"(f1y) : "r"(pre_a + 8u * (uint32_t)t));
              step(f0x, f0y);
              const uint32_t ka = kk;
              step(f1x, f1y);
              asm volatile("st.shared.u32 [%0], %1;" ::"r"(rec_a + 2u * (uint32_t)t), "r"(__byte_perm(ka, kk, 0x5410)) : "memory");
            }
            if (t < tn) { single(t); ++t; }
            if (tn < T) {  // the noise step (environments.py:25-36 with the redrawn intercept)
              uint32_t fx, fy, gj;
              asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(fx), "=r"(fy) : "r"(pre_a + 8u * (uint32_t)tn));
              asm volatile("ld.shared.u32 %0, [%1];" : "=r"(gj) : "r"(gj_a + sig4));
              kk = (gj & fx) | fy;
              const int k0 = (int)(kk & 0xff), k1 = (int)(kk >> 8);
              const uint32_t joint = __dp4a(kk, dp_b, 0u);
              const double aq0 = __dmul_rn(ab, scale_action(k0, A0, G.agent[0].action_lo, G.agent[0].action_hi));
              const double aq1 = __dmul_rn(ab, scale_action(k1, A1, G.agent[1].action_lo, G.agent[1].action_hi));
              const double na = nrec[k];
              const double pn = __dsub_rn(na, __dmul_rn(G.b, __dadd_rn(__dadd_rn(0.0, aq0), aq1)));
              const double np = pn > 0.0 ? pn : (pn != pn ? pn : 0.0);
              const double r0 = __dmul_rn(np, aq0), r1 = __dmul_rn(np, aq1);
              if (lane < 2) lg = __ddiv_rn(lane == 0 ? r0 : r1, Td);                      // trainer.py:65
              else if (lane < 4) lg = lutLog[4 * joint + lane];                           // trainer.py:66
              acc = __dadd_rn(acc, lg);
              const int ta0 = act_row(np, (float)G.agent[0].max_state, (float)G.agent[0].states);
              const int tu0 = upd_row(np, G.agent[0].max_state, (double)G.agent[0].states);
              const int ta1 = act_row(np, (float)G.agent[1].max_state, (float)G.agent[1].states);
              const int tu1 = upd_row(np, G.agent[1].max_state, (double)G.agent[1].states);
              __syncwarp();
              if (lane == 0) {
                nrec[k] = np;
                rowsW[NS + 1 + k] = (uint32_t)ta0 | ((uint32_t)tu0 << 8) | ((uint32_t)ta1 << 16) | ((uint32_t)tu1 << 24);
                GJ[NS + 1] = (uint32_t)grow[ta0] | ((uint32_t)grow[NR0 + 2 + ta1] << 8);  // the rollout only ever stands on the latest one
                rec[tn] = (uint16_t)kk;
              }
              __syncwarp();
              sig4 = 4u * (uint32_t)(NS + 1);
              t = tn + 1;
            }
          }
        }
        last_k = (int)kk;
      }
      __syncwarp();
      if (kNoise) {
        // states before every step, rebuilt lane-parallel from the action record; the state after a noise step is that
        // step's extra state
        for (int t = lane; t <= T; t += 32) {
          uint32_t s4 = sig4_start;
          if (t > 0) { const uint32_t kk = rec[t - 1]; s4 = nextS[__dp4a(kk, dp_b, 0u)]; }
          seq[t] = (uint8_t)(s4 >> 2);
        }
        __syncwarp();
        for (int k = lane; k < nK; k += 32) seq[nT[k] + 1] = (uint8_t)(NS + 1 + k);
        __syncwarp();
      }
      // compact rows of the state before step j (rowsW entry).  Noise-free, that state is where step j-1 led,
      // nextS[joint(rec[j-1])], and the episode's start state for j = 0; nextS holds 4 x state, the entry's byte offset.
      auto rows_before = [&](int j) -> uint32_t {
        if (kNoise) return rowsW[seq[j]];
        const uint32_t led = nextS[__dp4a((uint32_t)rec[j > 0 ? j - 1 : 0], dp_b, 0u)];  // loads, then a select: no branch
        return *reinterpret_cast<const uint32_t*>(reinterpret_cast<const unsigned char*>(rowsW) + (j > 0 ? led : sig4_start));
      };

      // optional per-step traces (parity runs only), lane-parallel
      if (p.trace_actions || p.trace_rewards || p.trace_prices) {
        const double ab = __ddiv_rn(G.a, G.b);
        for (int t = lane; t < T; t += 32) {
          const int k0 = rec[t] & 0xff, k1 = rec[t] >> 8, joint = k0 * A1 + k1;
          if (p.trace_actions) { p.trace_actions[(step0 + t) * 2] = k0; p.trace_actions[(step0 + t) * 2 + 1] = k1; }
          const int ks = kNoise && seq[t + 1] > NS ? (int)seq[t + 1] - NS - 1 : -1;  // noise step: its event record
          if (p.trace_rewards && ks >= 0) {  // environments.py:34 with the noise step's price
            p.trace_rewards[(step0 + t) * 2] = __dmul_rn(nrec[ks], __dmul_rn(ab, scale_action(k0, A0, G.agent[0].action_lo, G.agent[0].action_hi)));
            p.trace_rewards[(step0 + t) * 2 + 1] = __dmul_rn(nrec[ks], __dmul_rn(ab, scale_action(k1, A1, G.agent[1].action_lo, G.agent[1].action_hi)));
          } else if (p.trace_rewards) {
            p.trace_rewards[(step0 + t) * 2] = __dmul_rn(lutP[joint], lutAq[k0]);
            p.trace_rewards[(step0 + t) * 2 + 1] = __dmul_rn(lutP[joint], lutAq[A0 + k1]);
          }
          if (p.trace_prices && ks >= 0) {
            p.trace_prices[step0 + t] = nrec[ks];
          } else if (p.trace_prices) {
            const double aq0 = __dmul_rn(ab, scale_action(k0, A0, G.agent[0].action_lo, G.agent[0].action_hi));
            const double aq1 = __dmul_rn(ab, scale_action(k1, A1, G.agent[1].action_lo, G.agent[1].action_hi));
            const double pn = __dsub_rn(G.a, __dmul_rn(G.b, __dadd_rn(__dadd_rn(0.0, aq0), aq1)));
            p.trace_prices[step0 + t] = pn > 0.0 ? pn : (pn != pn ? pn : 0.0);
          }
        }
      }

      // ---- C: snapshot pass over the batch = the newest L_i transitions of the episode (buffers.py:12, agents.py:61-67):
      //      the stale old values (agents.py:67) of ALL transitions are read before any cell is written; visit counters
      //      and the dirty-row masks ride along.  Everything else a transition needs is expanded chunk by chunk below,
      //      which keeps the per-run scratch small (more runs resident per SM).
      unsigned dirty0a = 0, dirty0b = 0, dirty1a = 0, dirty1b = 0;  // written compact rows 0..63 of each agent
      bool dirty_all0 = false, dirty_all1 = false;
      // Agent 1's pass reads the rows word of each of its steps from the olds slot it then fills.  With equal batches (the
      // usual case) agent 0's pass visits the same steps and leaves it there, so the state is derived once per step.
      const bool pass_rows = L0 == L1;
      if (!pass_rows)
        for (int j = T - L1 + lane; j < T; j += 32) reinterpret_cast<uint32_t*>(olds + 2 * (j - (T - L1)) + 1)[0] = rows_before(j);
      for (int j = T - L0 + lane; j < T; j += 32) {
        const uint32_t rw = rows_before(j);
        const int k = rec[j] & 0xff, cu = (rw >> 8) & 0xff, jj = j - (T - L0);
        olds[2 * jj] = tab0[cu * A0 + k];
        if (pass_rows) reinterpret_cast<uint32_t*>(olds + 2 * jj + 1)[0] = rw;
        if (cnt0) atomicAdd(cnt0 + (size_t)table_row0(cu) * G.agent[0].row_stride + k, 1u);  // agents.py:76
        if (cu < 32) dirty0a |= 1u << cu; else if (cu < 64) dirty0b |= 1u << (cu - 32); else dirty_all0 = true;
      }
      for (int j = T - L1 + lane; j < T; j += 32) {
        const int k = rec[j] >> 8, cu = reinterpret_cast<const uint32_t*>(olds + 2 * (j - (T - L1)) + 1)[0] >> 24;
        olds[2 * (j - (T - L1)) + 1] = tab1[cu * A1 + k];
        if (cnt1) atomicAdd(cnt1 + (size_t)table_row1(cu) * G.agent[1].row_stride + k, 1u);
        if (cu < 32) dirty1a |= 1u << cu; else if (cu < 64) dirty1b |= 1u << (cu - 32); else dirty_all1 = true;
      }
      __syncwarp();

      // chunk expansion, lane-parallel: transition jj of agent ag -> (next-row byte offset, cell address, reward, (1-alpha)*old).
      // Noise-free, every lane calls it, a lane of half h taking transition jj = c0 + (lane & 15) (clamped to the batch: lanes
      // past its end repeat the last transition, and their countdown never reaches the store).  It loads the compact rows
      // after its step only: the rows before it are the rows after the previous transition, held by the lane below, and for
      // the first lane of a half they are carried over from the previous chunk (rw_carry: rows before transition c0 on entry,
      // before c0 + 16 on return).
      auto expand = [&](int jj, int ag, int La, double oma, uint32_t& rw_carry, uint32_t& row_off, uint32_t& cell_addr,
                        double2& v) {
        const int j = T - La + jj;
        const uint32_t kk = rec[j];
        uint32_t rw, rn;
        if (kNoise) {
          rw = rowsW[seq[j]];
          rn = rowsW[seq[j + 1]];
        } else {
          rn = *reinterpret_cast<const uint32_t*>(reinterpret_cast<const unsigned char*>(rowsW) + nextS[__dp4a(kk, dp_b, 0u)]);
          const uint32_t below = __shfl_up_sync(kFull, rn, 1, kLut2Chunk);
          rw = (lane & (kLut2Chunk - 1)) ? below : rw_carry;
          rw_carry = __shfl_sync(kFull, rn, kLut2Chunk - 1);
        }
        const int joint = (int)__dp4a(kk, dp_b, 0u);
        // the agent's bytes: k = byte ag of kk, update rows = byte 1 + 2 ag of a rows word (one PRMT each)
        const uint32_t sel_row = ag ? 0x4443u : 0x4441u;
        const int Aa = ag ? A1 : A0, k = (int)__byte_perm(kk, 0u, ag ? 0x4441u : 0x4440u);
        const int cu = (int)__byte_perm(rw, 0u, sel_row), cn = (int)__byte_perm(rn, 0u, sel_row);
        row_off = (uint32_t)(cn * Aa) * (uint32_t)sizeof(QT);
        cell_addr = (ag ? tab1_off : tab0_off) + (uint32_t)(cu * Aa + k) * (uint32_t)sizeof(QT);
        double rew = __dmul_rn(lutP[joint], lutAq[ag ? A0 + k : k]);
        if (kNoise && seq[j + 1] > NS) {  // a noise step: reward = its price x the agent's quantity (environments.py:34)
          const ThrlAgentSpec& sa = G.agent[ag];
          rew = __dmul_rn(nrec[(int)seq[j + 1] - NS - 1], __dmul_rn(__ddiv_rn(G.a, G.b), scale_action(k, Aa, sa.action_lo, sa.action_hi)));
        }
        v = make_double2(rew, __dmul_rn(oma, (double)olds[2 * jj + ag]));
        asm volatile("" : "+d"(v.x), "+d"(v.y), "+r"(cell_addr));  // computed here, not sunk into the update's loop
      };

      // ---- D: the sequential pass (agents.py:68-76).  The two agents' chains are independent: both rows are loaded
      //      before either cell is stored so the two dependency chains overlap.
      auto load_max = [&](uint32_t tab_lane_off, int A, bool in, uint32_t row_off) -> QT {
        const QT* row_lane = reinterpret_cast<const QT*>(smem + (tab_lane_off + row_off));
        if (kSmallA) return warp_max(row_lane[0]);                        // live table (:71)
        return lut2_row_max<QT, false>(row_lane, A, lane, in);
      };
      if (L0 == L1) {
        // Both agents in one instruction stream, lanes 0-15 carrying agent 0 and lanes 16-31 agent 1.  Lane i of each half
        // expands transition c0+i of its agent and keeps the cell address, reward and (1-alpha)*old in registers; only the
        // two next-row offsets of every transition go through shared memory (one uniform 8-byte load per iteration).  The
        // row maxima are warp reductions, so every lane evaluates :72-74 and the lane that owns transition j stores.
        const int li = lane & (kLut2Chunk - 1);
        uint32_t rw_carry = kNoise ? 0u : rows_before(T - L0);
        for (int c0 = 0; c0 < L0; c0 += kLut2Chunk) {
          const int n = L0 - c0 < kLut2Chunk ? L0 - c0 : kLut2Chunk;
          uint32_t row_off = 0, cell_addr = 0;
          double2 v = make_double2(0.0, 0.0);
          if (!kNoise) expand(min(c0 + li, L0 - 1), lane >> 4, L0, oma_h, rw_carry, row_off, cell_addr, v);
          else if (li < n) expand(c0 + li, lane >> 4, L0, oma_h, rw_carry, row_off, cell_addr, v);
          const uint32_t other = __shfl_xor_sync(kFull, row_off, 16);
          if (lane < n) *reinterpret_cast<uint2*>(smem + chunk_off + lane * 8) = make_uint2(row_off, other);
          __syncwarp();
          uint32_t ca = smem_base + chunk_off;
          int cd = li;  // iterations until this lane's transition is applied
          uint32_t mx_, my_;  // next-row offsets, loaded one iteration ahead (off the store -> load chain; the slot after the
                              // last transition of a full chunk is the 8-byte pad behind it)
          asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(mx_), "=r"(my_) : "r"(ca));
#pragma unroll 2
          for (int j = n; j > 0; --j, --cd) {
            const uint32_t ox = mx_, oy = my_;
            ca += 8u;
            asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(mx_), "=r"(my_) : "r"(ca));
            const QT mx0 = load_max(tab0_lane_off, A0, in0, ox);
            const QT mx1 = load_max(tab1_lane_off, A1, in1, oy);
            const double mx = (double)(hi_half ? mx1 : mx0);
            const double nv = __dadd_rn(v.y, __dmul_rn(alpha_h, __dadd_rn(v.x, __dmul_rn(gamma_h, mx))));  // :72-74
            if (cd == 0) *reinterpret_cast<QT*>(smem + cell_addr) = (QT)nv;                                 // :75
            __syncwarp();
          }
        }
      } else {
        for (int ag = 0; ag < 2; ++ag) {
          const int La = ag ? L1 : L0;
          const double alpha = hparam(ag, 0), gamma = hparam(ag, 1), oma = __dsub_rn(1.0, alpha);
          uint32_t rw_carry = kNoise || La == 0 ? 0u : rows_before(T - La);
          for (int c0 = 0; c0 < La; c0 += kLut2Chunk) {
            const int n = La - c0 < kLut2Chunk ? La - c0 : kLut2Chunk;
            uint32_t row_off = 0, cell_addr = 0;
            double2 v = make_double2(0.0, 0.0);
            const int li = lane & (kLut2Chunk - 1);  // lanes 16-31 repeat lanes 0-15 and never store
            if (!kNoise) expand(min(c0 + li, La - 1), ag, La, oma, rw_carry, row_off, cell_addr, v);
            else if (lane < n) expand(c0 + lane, ag, La, oma, rw_carry, row_off, cell_addr, v);
            if (lane < n) *reinterpret_cast<uint32_t*>(smem + chunk_off + lane * 8) = row_off;
            __syncwarp();
            for (int j = 0; j < n; ++j) {
              const uint32_t ro = *reinterpret_cast<const uint32_t*>(smem + chunk_off + j * 8);
              const double mx = (double)(ag ? load_max(tab1_lane_off, A1, in1, ro) : load_max(tab0_lane_off, A0, in0, ro));
              const double nv = __dadd_rn(v.y, __dmul_rn(alpha, __dadd_rn(v.x, __dmul_rn(gamma, mx))));  // :72-74
              if (lane == j) *reinterpret_cast<QT*>(smem + cell_addr) = (QT)nv;                          // :75
              __syncwarp();
            }
          }
        }
      }

      // ---- E: refresh the greedy cache of written rows, then the per-state greedy pairs
      {
        // lane = written row: a lane scans one row left to right for its first maximum (agents.py:88)
        auto scan_row = [&](const QT* row, int A) -> int {
          QT m = row[0];
          int g = 0;
#pragma unroll 4
          for (int k = 1; k < A; ++k) {
            const QT v = row[k];
            if (v > m) { m = v; g = k; }
          }
          return g;
        };
        // Rows 0..63 of both agents: the written ones (masks of C) are listed in the olds scratch, which D is done with,
        // agent 0's first.  A batch writes at most L0 + L1 <= 2T rows and olds holds 2T elements, so the list fits; one pass
        // of the warp covers 32 written rows of the two agents together (typically all of them) instead of two passes over
        // every compact row of each agent.
        const unsigned w0a = __reduce_or_sync(kFull, dirty0a), w0b = __reduce_or_sync(kFull, dirty0b);
        const unsigned w1a = __reduce_or_sync(kFull, dirty1a), w1b = __reduce_or_sync(kFull, dirty1b);
        const unsigned below = (1u << lane) - 1u;
        const int n0a = __popc(w0a), n0 = n0a + __popc(w0b), n1a = n0 + __popc(w1a), nd = n1a + __popc(w1b);
        uint8_t* dlist = reinterpret_cast<uint8_t*>(olds);
        if ((w0a >> lane) & 1u) dlist[__popc(w0a & below)] = (uint8_t)lane;
        if ((w0b >> lane) & 1u) dlist[n0a + __popc(w0b & below)] = (uint8_t)(32 + lane);
        if ((w1a >> lane) & 1u) dlist[n0 + __popc(w1a & below)] = (uint8_t)lane;
        if ((w1b >> lane) & 1u) dlist[n1a + __popc(w1b & below)] = (uint8_t)(32 + lane);
        __syncwarp();
        for (int i = lane; i < nd; i += 32) {  // selects, not a branch: lanes of both agents scan together
          const bool ag = i >= n0;
          const int c = dlist[i], A = ag ? A1 : A0;
          grow[(ag ? NR0 + 2 : 0) + c] = (uint8_t)scan_row((ag ? tab1 : tab0) + c * A, A);
        }
        // rows from 64 on are not in the masks: all of them when the batch wrote any
        if (__any_sync(kFull, dirty_all0))
          for (int c = 64 + lane; c < NR0 + 2; c += 32) grow[c] = (uint8_t)scan_row(tab0 + c * A0, A0);
        if (__any_sync(kFull, dirty_all1))
          for (int c = 64 + lane; c < NR1 + 2; c += 32) grow[NR0 + 2 + c] = (uint8_t)scan_row(tab1 + c * A1, A1);
        __syncwarp();
        if (kNoise && sig4 > 4u * (uint32_t)NS) {  // the episode ended on a noise step: its state becomes the next episode's state NS
          if (lane == 0) rowsW[NS] = rowsW[NS + nK];
          noise_price = nrec[nK - 1];
          sig4 = 4u * (uint32_t)NS;
          __syncwarp();
        } else if (kNoise) {
          noise_price = -1.0;
        }
        for (int s = lane; s <= NS; s += 32) {
          const uint32_t rw = rowsW[s];
          GJ[s] = (uint32_t)grow[rw & 0xff] | ((uint32_t)grow[NR0 + 2 + ((rw >> 16) & 0xff)] << 8);
        }
      }
      // epsilon decay, every epoch (agents.py:78)
      {
        const double epsend0 = hparam(0, 2), epsstep0 = hparam(0, 3), epsend1 = hparam(1, 2), epsstep1 = hparam(1, 3);
        eps0 = __dadd_rn(epsend0, __dmul_rn(__dsub_rn(eps0, epsend0), epsstep0));
        eps1 = __dadd_rn(epsend1, __dmul_rn(__dsub_rn(eps1, epsend1), epsstep1));
      }
      // logs and statistics: lane 0,1 = rewards_log[e, 0..1], lane 2,3 = actions_log[e, 0..1]
      if (lane < 4) {
        const int ag = lane & 1;
        if (r < p.n_log_runs) {
          double* dst = lane < 2 ? p.rewards_log : p.actions_log;
          if (dst) dst[(r * E + e) * 2 + ag] = acc;
        }
        if (p.stats) {
          unsigned long long* s4 = reinterpret_cast<unsigned long long*>(p.stats) + ((size_t)e * 2 + ag) * THRL_STATS_K + (lane < 2 ? 0 : 2);
          atomicAdd(s4 + 0, (unsigned long long)fx_round(__dmul_rn(acc, THRL_STATS_SCALE_SUM)));
          atomicAdd(s4 + 1, (unsigned long long)fx_round(__dmul_rn(__dmul_rn(acc, acc), THRL_STATS_SCALE_SQ)));
        }
      }
      __syncwarp();
    }

    // ---- write the run back: only the staged rows can have changed
    for (int c = 0; c < NR0 + 2; ++c) {
      const int row = table_row0(c);
      if (row >= 0) for (int k = lane; k < A0; k += 32) qg0[(size_t)row * G.agent[0].row_stride + k] = tab0[c * A0 + k];
    }
    for (int c = 0; c < NR1 + 2; ++c) {
      const int row = table_row1(c);
      if (row >= 0) for (int k = lane; k < A1; k += 32) qg1[(size_t)row * G.agent[1].row_stride + k] = tab1[c * A1 + k];
    }
    if (lane == 0) {
      p.eps[r * 2] = eps0;
      p.eps[r * 2 + 1] = eps1;
      if (kNoise && noise_price >= 0.0) {
        p.price[r] = noise_price;
      } else if (last_k >= 0) {  // environments.py:36 self.state = price of the last step
        const double ab = __ddiv_rn(G.a, G.b);
        const double aq0 = __dmul_rn(ab, scale_action(last_k & 0xff, A0, G.agent[0].action_lo, G.agent[0].action_hi));
        const double aq1 = __dmul_rn(ab, scale_action(last_k >> 8, A1, G.agent[1].action_lo, G.agent[1].action_hi));
        const double pn = __dsub_rn(G.a, __dmul_rn(G.b, __dadd_rn(__dadd_rn(0.0, aq0), aq1)));
        p.price[r] = pn > 0.0 ? pn : (pn != pn ? pn : 0.0);
      }
    }
    __syncwarp();
  }
}

}  // namespace thrl
