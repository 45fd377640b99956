// thrl.cu — C ABI (include/thrl.h) of the B200-native th_rl hot path: validation, shared-memory layout, launches.
// Compile: nvcc -gencode arch=compute_100a,code=sm_100a --fmad=false -lineinfo (see th_rl_b200/build.py).
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <math.h>
#include <stdlib.h>

#include <algorithm>
#include <array>
#include <cmath>
#include <atomic>
#include <map>
#include <memory>
#include <mutex>
#include <set>
#include <vector>

#include "thrl_device.cuh"
#include "thrl_scan_generic.cuh"
#include "thrl_scan_hbm.cuh"
#include "thrl_scan_lut2.cuh"
#include "thrl_scan_lpc.cuh"
#include "thrl_scan_mixed.cuh"
#include "thrl_scan_pwl.cuh"
#include "thrl_scan_pwc.cuh"
#include "thrl_aux_kernels.cuh"

namespace {

thread_local char g_err[512] = "";
thread_local long long g_last_wave = 0;  // runs resident at once in this thread's latest scan launch (thrl_last_wave_runs)
thread_local const char* g_last_kernel = "";  // scan kernel of this thread's latest thrl_qtable_scan (thrl_last_kernel)
std::atomic<long long> g_launches{0};

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
#define CUDA_TRY(expr)                                                                              \
  do {                                                                                              \
    cudaError_t e_ = (expr);                                                                        \
    if (e_ != cudaSuccess) return fail(THRL_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(e_));     \
  } while (0)

inline int align_up(int x, int a) { return (x + a - 1) / a * a; }

struct DeviceInfo {
  int sms = 0, smem_optin = 0, cc_major = 0;
};
int device_info(DeviceInfo* d) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return fail(THRL_ERR_NO_DEVICE, "no CUDA device (there is no CPU fallback)");
  CUDA_TRY(cudaDeviceGetAttribute(&d->sms, cudaDevAttrMultiProcessorCount, dev));
  CUDA_TRY(cudaDeviceGetAttribute(&d->smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  CUDA_TRY(cudaDeviceGetAttribute(&d->cc_major, cudaDevAttrComputeCapabilityMajor, dev));
  if (d->cc_major != 10) return fail(THRL_ERR_NO_DEVICE, "device is sm_%d0, this library is built for sm_100a only", d->cc_major);
  return THRL_OK;
}

double h_scale(int k, int actions, double lo, double hi);
int h_act_row(double price, double max_state, int states);
int h_upd_row(double price, double max_state, int states);

int validate_layout(ThrlGame* G) {
  if (!G) return fail(THRL_ERR_BAD_ARGS, "game is NULL");
  if (G->n_agents < 1 || G->n_agents > THRL_MAX_AGENTS)
    return fail(THRL_ERR_BAD_CONFIG, "n_agents=%d outside 1..%d", G->n_agents, THRL_MAX_AGENTS);
  if (G->max_steps < 1) return fail(THRL_ERR_BAD_CONFIG, "max_steps=%d", G->max_steps);
  if (!(G->b == G->b) || G->b == 0.0) return fail(THRL_ERR_BAD_CONFIG, "b must be non-zero");
  long long off = 0, moff = 0;
  int ring = 0, regular = 1;
  // tables that stay in HBM are padded: rows, table offsets and the run stride are multiples of 4 elements (include/thrl.h)
  long long cells = 0;
  for (int i = 0; i < G->n_agents; ++i)
    if (G->agent[i].kind == THRL_AGENT_QTABLE && G->agent[i].states >= 1 && G->agent[i].actions >= 1)
      cells += (long long)(G->agent[i].states + 1) * G->agent[i].actions;
  const bool padded = cells * 4 >= THRL_PAD_THRESHOLD_BYTES;
  for (int i = 0; i < G->n_agents; ++i) {
    ThrlAgentSpec* s = &G->agent[i];
    G->mlp_buffer_len[i] = 0;
    s->row_stride = 0;
    s->reserved_ = 0;
    if (s->actions < 2 || s->actions > THRL_MAX_ACTIONS)
      return fail(THRL_ERR_BAD_CONFIG, "agent %d: actions=%d outside 2..%d", i, s->actions, THRL_MAX_ACTIONS);
    if (s->capacity < 0 || s->min_memory < 0) return fail(THRL_ERR_BAD_CONFIG, "agent %d: negative capacity/min_memory", i);
    const int T = G->max_steps, mm = s->min_memory > 0 ? s->min_memory : 1;
    long long need = (long long)T * ((mm + T - 1) / T);
    if (need > s->capacity) need = s->capacity;
    if (s->kind == THRL_AGENT_REINFORCE || s->kind == THRL_AGENT_ACTORCRITIC || s->kind == THRL_AGENT_CAC) {
      if (s->states != 1) return fail(THRL_ERR_BAD_CONFIG, "agent %d: states=%d for an MLP agent, the environment's state is one number", i, s->states);
      if (s->hidden < 1 || s->hidden > 1024) return fail(THRL_ERR_BAD_CONFIG, "agent %d: hidden=%d outside 1..1024", i, s->hidden);
      if (!(s->entropy == s->entropy)) return fail(THRL_ERR_BAD_CONFIG, "agent %d: entropy coefficient is NaN", i);
      const bool ac = s->kind != THRL_AGENT_REINFORCE;  // 4-word transitions (new_state kept)
      const long long P = s->kind == THRL_AGENT_CAC ? 5LL * s->hidden + 3
                                                    : 2LL * s->hidden + (long long)s->actions * s->hidden + s->actions + (s->kind == THRL_AGENT_ACTORCRITIC ? s->hidden + 1 : 0);
      G->mlp_buffer_len[i] = s->min_memory <= s->capacity ? (int32_t)need : 0;
      s->mlp_offset = moff;
      s->table_offset = 0;
      moff += 3 * P + THRL_MLP_HEADER_WORDS + (ac ? 4LL : 3LL) * G->mlp_buffer_len[i];
      continue;
    }
    if (s->kind != THRL_AGENT_QTABLE) return fail(THRL_ERR_BAD_CONFIG, "agent %d: unknown kind %d", i, s->kind);
    if (s->states < 1 || s->states > 65534) return fail(THRL_ERR_BAD_CONFIG, "agent %d: states=%d outside 1..65534", i, s->states);
    // the reference raises IndexError on the first encode whose row exceeds `states` (agents.py:88).  Prices never exceed a
    // (environments.py:28-32: new_a <= a), so the largest reachable row is the encode of a itself -- by either encode, the
    // float32 one of sample_action or the float64 one of train_net; a slightly above max_state may still round into the table
    if (!(s->max_state > 0.0) || !(G->a == G->a))
      return fail(THRL_ERR_BAD_CONFIG, "agent %d: max_state=%g", i, s->max_state);
    if (h_act_row(G->a, s->max_state, s->states) > s->states || h_upd_row(G->a, s->max_state, s->states) > s->states)
      return fail(THRL_ERR_BAD_CONFIG, "agent %d: a=%g with max_state=%g encodes to a row past the table's %d (reference: IndexError)", i,
                  G->a, s->max_state, s->states);
    s->table_offset = off;
    s->mlp_offset = 0;
    s->row_stride = padded ? align_up(s->actions, 4) : s->actions;
    off += (long long)(s->states + 1) * s->row_stride;
    if (s->min_memory <= s->capacity) {
      if (need > ring) ring = (int)need;
      if (s->min_memory > T) regular = 0;
    }
  }
  if (off >= (1LL << 31) || moff >= (1LL << 31)) return fail(THRL_ERR_UNSUPPORTED, "one run's tables hold %lld elements (limit 2^31-1)", off);
  G->run_stride = off;
  G->mlp_stride = moff;
  G->ring_len = ring;
  G->regular = regular;
  return THRL_OK;
}

long long ring_bytes(const ThrlGame* G) {
  const long long Hp = (G->ring_len > 0 ? G->ring_len : 1) + 1;
  long long b = (long long)sizeof(thrl::RingHeader) + Hp * 8 + (long long)G->n_agents * Hp;
  return (b + 15) / 16 * 16;
}

// Fills the shared-memory layout of ScanParams; returns bytes per warp slot.
void plan_generic(thrl::ScanParams* p, bool smem_tables, size_t elem) {
  const ThrlGame& G = p->game;
  const int n = G.n_agents, T = G.max_steps, Hp = p->Hp;
  int lut = 0, rows = 0;
  // rows the price can reach: price <= a - a * sum_i min(action_range_i) (environments.py:25-32 with new_a <= a), +2 rows
  // of slack for rounding; the call's initial price may lie above and is handled uncached
  double lo_sum = 0.0;
  bool bounded = G.a >= 0.0 && G.b > 0.0;
  for (int i = 0; i < n; ++i) {
    const double lo = G.agent[i].action_lo < G.agent[i].action_hi ? G.agent[i].action_lo : G.agent[i].action_hi;
    if (!(lo >= 0.0)) bounded = false;
    lo_sum += lo;
  }
  for (int i = 0; i < n; ++i) {
    int cap = G.agent[i].states + 1;
    if (bounded) {
      double pmax = G.a - G.a * lo_sum;
      if (pmax < 0.0) pmax = 0.0;
      const double rmax = pmax / G.agent[i].max_state * (double)G.agent[i].states + 2.5;
      if (rmax < (double)cap) cap = (int)rmax;
    }
    p->gcap[i] = cap;
    lut += G.agent[i].actions;
    rows += cap;
  }
  p->lut_total = lut;
  p->rows_total = rows;
  int amax = 0;
  for (int i = 0; i < n; ++i) if (G.agent[i].actions > amax) amax = G.agent[i].actions;
  p->quarter = (n <= 8 && amax <= 128 && !getenv("THRL_NO_QUARTER")) ? 1 : 0;
  p->qchunks = (amax + 7) / 8;
  {  // columns per lane the kernel dispatches to (thrl_scan_generic.cuh); qfull: only the last of them can lie beyond a row's end
    const int nc = p->qchunks <= 4 ? 4 : (p->qchunks <= 8 ? 8 : (p->qchunks <= 13 ? 13 : 16));
    int amin = amax;
    for (int i = 0; i < n; ++i) if (G.agent[i].actions < amin) amin = G.agent[i].actions;
    p->qfull = (amin >= 8 * (nc - 1) && !getenv("THRL_NO_QFULL")) ? 1 : 0;
  }
  p->cta_bytes = align_up(2 * lut * 8, 16);
  int o = 0;
  p->off_tab = o;
  if (smem_tables) o += align_up((int)(G.run_stride * (long long)elem), 16);
  p->off_P = o;    o += align_up(Hp * 8, 16);
  p->off_newa = o; o += p->noisy ? align_up(T * 8, 16) : 0;
  p->off_hp = o;   o += align_up(n * 5 * 8, 16);
  p->old_stride = align_up(Hp, 4);
  p->off_old = o;  o += align_up(n * p->old_stride * (int)elem, 16);
  p->off_pre = o;  o += align_up(T * n * 2, 16);
  p->row_stride = align_up(Hp + 1, 8);
  p->off_row = o;  o += align_up(n * p->row_stride * 2, 16);
  p->off_des = o;  o += align_up(n * 4 * 4, 16);
  p->off_act = o;  o += align_up(n * Hp, 16);
  p->off_g = o;    o += align_up(rows, 16);
  p->warp_bytes = o;
}

template <typename T>
int launch_generic(thrl::ScanParams& p, const DeviceInfo& dev, cudaStream_t stream) {
  const ThrlGame& G = p.game;
  const long long tab_bytes = G.run_stride * (long long)sizeof(T);
  // Tables go to shared memory when at least 4 runs fit next to each other on an SM; otherwise they stay in HBM.
  bool smem_tables = false;
  if (tab_bytes < dev.smem_optin / 4) {
    plan_generic(&p, true, sizeof(T));
    smem_tables = (dev.smem_optin - p.cta_bytes) / p.warp_bytes >= 4;
  }
  if (!smem_tables) plan_generic(&p, false, sizeof(T));
  int warps = (dev.smem_optin - p.cta_bytes) / p.warp_bytes;
  if (warps < 1) return fail(THRL_ERR_UNSUPPORTED, "one run needs %d B of shared memory (> %d B)", p.warp_bytes + p.cta_bytes, dev.smem_optin);
  if (warps > (smem_tables ? 32 : 16)) warps = smem_tables ? 32 : 16;
  // every warp plays whole runs one after another: spread the runs evenly over the rounds that are needed anyway
  int grid = dev.sms;
  {
    const long long slots = (long long)dev.sms * warps;
    const long long rounds = (p.n_runs + slots - 1) / slots;
    const long long per_round = (p.n_runs + rounds - 1) / rounds;
    warps = (int)((per_round + dev.sms - 1) / dev.sms);
    if (warps < 1) warps = 1;
    grid = (int)((per_round + warps - 1) / warps);
    if (grid > dev.sms) grid = dev.sms;
  }
  const size_t smem = (size_t)p.cta_bytes + (size_t)warps * p.warp_bytes;
  auto kern = smem_tables ? thrl::qtable_scan_generic<T, true> : thrl::qtable_scan_generic<T, false>;
  CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  g_last_kernel = "generic";
  g_last_wave = (long long)grid * warps;
  kern<<<grid, warps * 32, smem, stream>>>(p);
  CUDA_TRY(cudaGetLastError());
  g_launches.fetch_add(1);
  return THRL_OK;
}

// ------------------------------------------------------------------------------------------------ HBM-resident tables
// Fills p (per-agent constants + shared-memory layout) when thrl_scan_hbm.cuh plays the game; *warps = runs resident per CTA.
bool plan_hbm(thrl::HbmParams* p, size_t elem, const DeviceInfo& dev, int* warps) {
  const ThrlGame& G = p->game;
  const int n = G.n_agents, T = G.max_steps, esz = (int)elem;
  if (G.mlp_stride > 0 || !G.regular || T > thrl::kHbmMaxT || G.run_stride % 4) return false;
  if (G.run_stride * (long long)elem < THRL_PAD_THRESHOLD_BYTES) return false;  // small tables are staged in shared memory
  int lut = 0, rows = 0, rowbytes = 0;
  double lo_sum = 0.0;
  bool bounded = G.a >= 0.0 && G.b > 0.0;
  for (int i = 0; i < n; ++i) {
    const ThrlAgentSpec& s = G.agent[i];
    if (s.kind != THRL_AGENT_QTABLE || s.row_stride % 4 || s.table_offset % 4 || s.actions > 128) return false;
    const double lo = s.action_lo < s.action_hi ? s.action_lo : s.action_hi;
    if (!(lo >= 0.0)) bounded = false;
    lo_sum += lo;
  }
  p->ncls = 0;
  for (int i = 0; i < n; ++i) {
    const ThrlAgentSpec& s = G.agent[i];
    // rows the price can reach: price <= a - a * sum_i min(action_range_i) (environments.py:25-32 with new_a <= a), +2 rows
    // of slack for rounding; the call's initial price may lie above and is handled uncached
    int cap = s.states + 1;
    if (bounded) {
      double pmax = G.a - G.a * lo_sum;
      if (pmax < 0.0) pmax = 0.0;
      const double rmax = pmax / s.max_state * (double)s.states + 2.5;
      if (rmax < (double)cap) cap = (int)rmax;
    }
    p->gcap[i] = cap;
    p->goff[i] = rows;
    p->L[i] = s.min_memory > s.capacity ? 0 : (T < s.capacity ? T : s.capacity);
    rows += cap;
    // agents with the same action grid share one action LUT (AQ / XT)
    p->lut_owner[i] = i;
    for (int j = 0; j < i; ++j)
      if (G.agent[j].actions == s.actions && G.agent[j].action_lo == s.action_lo && G.agent[j].action_hi == s.action_hi) {
        p->lut_owner[i] = p->lut_owner[j];
        break;
      }
    if (p->lut_owner[i] == i) {
      p->loff[i] = lut;
      lut += s.actions;
    } else {
      p->loff[i] = p->loff[p->lut_owner[i]];
    }
    if (s.row_stride * esz > rowbytes) rowbytes = s.row_stride * esz;
    // state class: agents whose float64 encode (max_state, states) and batch (its length) coincide see the same rows
    p->cls_of[i] = -1;
    if (p->L[i] > 0) {
      for (int j = 0; j < i && p->cls_of[i] < 0; ++j)
        if (p->L[j] == p->L[i] && G.agent[j].states == s.states && G.agent[j].max_state == s.max_state) p->cls_of[i] = p->cls_of[j];
      if (p->cls_of[i] < 0) p->cls_of[i] = p->ncls++;
    }
  }
  for (int c = 0, k = 0; c < p->ncls; ++c) {
    p->cls_beg[c] = k;
    for (int i = 0; i < n; ++i)
      if (p->cls_of[i] == c) p->cls_agent[k++] = i;
    p->cls_na[c] = k - p->cls_beg[c];
  }
  p->lut_total = lut;
  p->rows_total = rows;
  p->nch_max = rowbytes / 16;
  p->Tp = align_up(T, 4);
  p->Sp = align_up(T + 1, 4);
  p->cta_bytes = align_up(2 * lut * 8 + n * thrl::kHbmAgc * 4, 128);
  const char* gmode = getenv("THRL_HBM_GATHER");  // reg (default) | bulk | ldg
  p->staged = (gmode && (strcmp(gmode, "bulk") == 0 || strcmp(gmode, "ldg") == 0)) ? 1 : 0;
  p->bulk = (gmode && strcmp(gmode, "ldg") == 0) ? 0 : 1;
  p->pf_dist = 2;
  if (const char* f = getenv("THRL_HBM_PF")) p->pf_dist = atoi(f) < 0 ? 0 : (atoi(f) > 16 ? 16 : atoi(f));
  const int Tp = p->Tp, Sp = p->Sp, nc = p->ncls > 0 ? p->ncls : 1;
  auto layout = [&](int nb, int lpr_shift) {
    const int lpr = 1 << lpr_shift, rb = 32 >> lpr_shift;
    // a quarter-warp reads 8 / lpr rows x lpr consecutive 16-byte chunks (8 rows x 1 chunk each for lpr = 1): distinct
    // banks when the slot stride is = lpr (mod 8) chunks
    int chunks = rowbytes / 16;
    while (chunks % 8 != lpr % 8) ++chunks;
    p->slot_bytes = chunks * 16;
    p->lpr_shift = lpr_shift;
    int o = 0;
    p->off_bar = o;   o += p->staged ? thrl::kHbmMaxNb * 8 : 0;
    p->off_g = o;     o += align_up(rows, 16);
    p->off_P = o;     o += align_up((T + 1) * 8, 16);
    p->off_hp = o;    o += align_up(n * 5 * 8, 16);
    p->off_miss = o;  o += 2 * THRL_MAX_AGENTS;
    p->off_srow = o;  o += align_up(nc * Sp * 2, 16);
    p->off_rs = o;    o += align_up(nc * Sp, 16);
    p->off_next = o;  o += align_up(nc * Sp, 16);
    p->off_dl = o;    o += align_up(nc * Sp, 16);
    p->off_act = o;   o += align_up(n * Tp, 16);
    p->off_cur = o;   o += align_up(n * Tp * esz, 16);
    p->off_canon = o; o += align_up(n * Tp, 16);
    p->off_nextc = o; o += align_up(n * Tp, 16);
    p->off_bm = o;    o += align_up(n * Sp * esz, 16);
    p->off_stage = o;
    p->off_pre = o;
    p->off_newa = o + align_up(T * n, 16);
    p->off_rq = o;
    p->off_mask = o;
    const int draws = align_up(T * n, 16) + (p->noisy ? T * 8 : 0);
    const int ring = p->staged ? nb * rb * p->slot_bytes : 32 * 16;  // register landing: the column masks of one batch
    int region = std::max(ring, std::max(draws, n * 8));
    region = align_up(region, 16);
    p->seg = region / (n * 8) < T ? region / (n * 8) : T;  // steps whose reward / max_steps fit the region at a time
    o += region;
    p->nb = nb;
    p->warp_bytes = align_up(o, 16);
    return p->warp_bytes;
  };
  const int avail = dev.smem_optin - p->cta_bytes;
  int w;
  if (!p->staged) {
    // Rows pass through L1 lines on their way to the registers: keep the CTA within the 196 KB shared-memory carve-out so that
    // 60 KB of L1 are left for the loads in flight (measured on the C4 shape: 12 resident runs per SM reach 5.8e9 agent-steps/s,
    // 13 -- which need the 228 KB carve-out -- 4.1e9).
    const int carve = 196 * 1024 - 1024;  // the driver reserves 1 KB per CTA
    const int budget = (avail < carve - p->cta_bytes ? avail : carve - p->cta_bytes);
    w = budget / layout(1, 1);
  } else {
    int lpr_shift = 1;  // two lanes per staged row, 16 rows per batch
    if (const char* f = getenv("THRL_HBM_LPR")) {
      const int v = atoi(f);
      if (v == 1) lpr_shift = 0; else if (v == 2) lpr_shift = 1; else if (v == 4) lpr_shift = 2; else if (v == 8) lpr_shift = 3;
    }
    while (lpr_shift < 3 && avail / layout(2, lpr_shift) < 1) ++lpr_shift;  // smaller batches when even two do not fit
    int nb = 2;
    if (avail / layout(nb, lpr_shift) < 1) nb = 1;
    w = avail / layout(nb, lpr_shift);
    if (w >= 1) {  // the rounds of the persistent grid are fixed by what fits; a deeper ring that still fits them costs nothing
      if (w > thrl::kHbmMaxWarps) w = thrl::kHbmMaxWarps;
      const long long slots = (long long)dev.sms * w;
      const long long rounds = (p->n_runs + slots - 1) / slots;
      const long long per_round = (p->n_runs + rounds - 1) / rounds;
      int wneed = (int)((per_round + dev.sms - 1) / dev.sms);
      if (wneed < 1) wneed = 1;
      const char* force = getenv("THRL_HBM_NB");
      if (force && atoi(force) >= 1 && atoi(force) <= thrl::kHbmMaxNb) {
        nb = atoi(force);
        if (avail / layout(nb, lpr_shift) < 1) return false;
      } else {
        while (nb < thrl::kHbmMaxNb && nb < 4 && (long long)layout(nb + 1, lpr_shift) * wneed <= avail) ++nb;
        layout(nb, lpr_shift);
      }
      w = avail / p->warp_bytes;
    }
  }
  if (w < 1) return false;
  if (w > (p->staged ? thrl::kHbmMaxWarps : thrl::kHbmRegWarps)) w = p->staged ? thrl::kHbmMaxWarps : thrl::kHbmRegWarps;
  if (const char* f = getenv("THRL_HBM_WARPS"))
    if (atoi(f) >= 1 && atoi(f) < w) w = atoi(f);
  *warps = w;
  // Dynamic schedule (thrl_scan_hbm.cuh): only where the static rounds leave slots idle -- more than one round, not a whole
  // number of them -- and the call is long enough for ~100-epoch tasks (a task starts with a cold greedy cache).  Register landing
  // only.  THRL_HBM_CHUNK = number of tasks per run (0 / 1: static schedule), for tests and comparisons.
  p->nchunk = 1;
  p->echunk = 0;
  p->off_q = p->cta_bytes;
  {
    const long long slots = (long long)dev.sms * w;
    int nchunk = 1;
    if (!p->staged && p->n_runs > slots && p->n_runs % slots != 0 && p->E >= 100) {
      // Cost model fitted on the C4 shape (one round of w resident runs per SM takes ~ 0.58 + 0.035 w of a 12-run round; a task
      // pays ~2 % of a run's chunk for its cold greedy cache): static = rounds x round time at the balanced residency; dynamic
      // with c tasks per run = ceil(runs per CTA x c / w) / c rounds at full residency.  Dynamic only when it wins by 5 %.
      const long long rounds = (p->n_runs + slots - 1) / slots;
      const double wbal = (double)((p->n_runs + rounds - 1) / rounds) / dev.sms;
      const double full = 0.58 + 0.035 * w;
      const double stat = (double)rounds * (0.58 + 0.035 * wbal) / full;
      const long long nloc = (p->n_runs + dev.sms - 1) / dev.sms;
      double best = stat * 0.95;
      for (int c = 2; c <= 8 && p->E / c >= 50; ++c) {
        const double dyn = (double)((nloc * c + w - 1) / w) / c * (1.0 + 0.02 * c);
        if (dyn < best) { best = dyn; nchunk = c; }
      }
    }
    if (const char* f = getenv("THRL_HBM_CHUNK")) nchunk = p->staged ? 1 : atoi(f);
    if (nchunk > p->E) nchunk = p->E;
    if (nchunk > 1) {
      const int grid = p->n_runs < dev.sms ? (int)p->n_runs : dev.sms;
      const long long nloc = (p->n_runs + grid - 1) / grid;
      const int qbytes = align_up(16 + 4 * (int)nloc, 128);
      if (nloc * nchunk < (1LL << 30) && p->cta_bytes + qbytes + (long long)w * p->warp_bytes <= dev.smem_optin) {
        p->nchunk = nchunk;
        p->echunk = (p->E + nchunk - 1) / nchunk;
        p->cta_bytes += qbytes;
      }
    }
  }
  return true;
}

template <typename QT>
int launch_hbm(thrl::HbmParams& p, int warps, const DeviceInfo& dev, cudaStream_t stream) {
  int grid = dev.sms;
  const long long capacity = (long long)dev.sms * warps;  // runs resident at once when the launch is large enough
  {  // every warp plays whole runs one after another: spread the runs evenly over the rounds that are needed anyway
    const long long slots = (long long)dev.sms * warps;
    const long long rounds = (p.n_runs + slots - 1) / slots;
    const long long per_round = (p.n_runs + rounds - 1) / rounds;
    if (p.nchunk > 1) {  // dynamic schedule: every CTA at full residency, tasks from the CTA's queue
      grid = p.n_runs < dev.sms ? (int)p.n_runs : dev.sms;
      const long long nloc = (p.n_runs + grid - 1) / grid;
      if (nloc * p.nchunk < warps) warps = (int)(nloc * p.nchunk);
      p.per_round = (long long)grid * warps;
    } else {
      warps = (int)((per_round + dev.sms - 1) / dev.sms);
      if (warps < 1) warps = 1;
      grid = per_round < dev.sms ? (int)per_round : dev.sms;  // partial warps of a round are spread over all SMs (slot = warp * grid + cta)
      p.per_round = per_round;
    }
  }
  const size_t smem = (size_t)p.cta_bytes + (size_t)warps * p.warp_bytes;
  auto kern = p.staged ? thrl::qtable_scan_hbm<QT, true> : (p.nchunk > 1 ? thrl::qtable_scan_hbm<QT, false, true> : thrl::qtable_scan_hbm<QT, false>);
  CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  g_last_kernel = "hbm";
  g_last_wave = capacity;
  kern<<<grid, warps * 32, smem, stream>>>(p);
  CUDA_TRY(cudaGetLastError());
  g_launches.fetch_add(1);
  return THRL_OK;
}

// ------------------------------------------------------------------------------------------------ LUT2 planning
// Host restatement of the per-joint-action price and its encodes; compiled with -ffp-contract=off, every operation is
// the same IEEE operation the device (and the reference) performs.
double h_scale(int k, int actions, double lo, double hi) {
  double d = (double)k / ((double)actions - 1.0);
  d = d * (hi - lo);
  return d + lo;
}
int h_act_row(double price, double max_state, int states) {
  float x = (float)price / (float)max_state;
  x = x * (float)states;
  return (int)rintf(x);
}
int h_upd_row(double price, double max_state, int states) {
  double x = price / max_state;
  x = x * (double)states;
  return (int)rint(x);
}

// Returns true and fills p (structure + layout) when the specialised kernel applies; *warps = runs resident per CTA.
bool plan_lut2(thrl::Lut2Params* p, bool noisy, size_t elem, int smem_optin, int* warps) {
  const ThrlGame& G = p->game;
  if (G.n_agents != 2 || !G.regular) return false;
  const int A0 = G.agent[0].actions, A1 = G.agent[1].actions, T = G.max_steps;
  if (A0 > 255 || A1 > 255 || A0 * A1 > thrl::kLut2MaxJoint || T > 32767) return false;
  // demand noise: the redrawn intercept lies in [0.7 a, a] (environments.py:28-31), so with non-negative quantities the price
  // stays in [0, a - a * (lo_0 + lo_1)]: every row up to that price's row is staged and a compact row is its table row
  int rmax[2] = {0, 0};
  if (noisy) {
    if (!(G.a > 0.0) || !(G.b > 0.0) || T > 200) return false;
    double lo_sum = 0.0;
    for (int a = 0; a < 2; ++a) {
      const double lo = std::fmin(G.agent[a].action_lo, G.agent[a].action_hi);
      if (!(lo >= 0.0)) return false;
      lo_sum += lo;
    }
    double pmax = G.a - G.a * lo_sum;
    if (!(pmax >= 0.0)) pmax = 0.0;
    for (int a = 0; a < 2; ++a) {
      const double r = pmax / G.agent[a].max_state * (double)G.agent[a].states + 2.5;
      rmax[a] = r < (double)G.agent[a].states ? (int)r : G.agent[a].states;
    }
  }
  p->noisy = noisy ? 1 : 0;
  const int J = A0 * A1;
  const double ab = G.a / G.b;
  std::map<std::array<int, 4>, int> ids;
  std::vector<std::array<int, 4>> tuples;
  std::vector<int> state_of(J);
  for (int j = 0; j < J; ++j) {
    const int k0 = j / A1, k1 = j % A1;
    const double aq0 = ab * h_scale(k0, A0, G.agent[0].action_lo, G.agent[0].action_hi);
    const double aq1 = ab * h_scale(k1, A1, G.agent[1].action_lo, G.agent[1].action_hi);
    double Q = 0.0 + aq0;
    Q = Q + aq1;
    const double pn = G.a - G.b * Q;
    const double price = pn > 0.0 ? pn : (pn != pn ? pn : 0.0);
    if (price != price) return false;
    std::array<int, 4> t = {h_act_row(price, G.agent[0].max_state, G.agent[0].states),
                            h_upd_row(price, G.agent[0].max_state, G.agent[0].states),
                            h_act_row(price, G.agent[1].max_state, G.agent[1].states),
                            h_upd_row(price, G.agent[1].max_state, G.agent[1].states)};
    auto it = ids.find(t);
    if (it == ids.end()) {
      it = ids.emplace(t, (int)tuples.size()).first;
      tuples.push_back(t);
    }
    state_of[j] = it->second;
  }
  const int NS = (int)tuples.size();
  if (NS > thrl::kLut2MaxStates) return false;
  std::set<int> rows[2];
  for (auto& t : tuples) { rows[0].insert(t[0]); rows[0].insert(t[1]); rows[1].insert(t[2]); rows[1].insert(t[3]); }
  if (noisy) {
    if (NS + 1 + T > 255) return false;  // state ids of an episode (lattice, initial, one per noise step) fit a byte
    for (int a = 0; a < 2; ++a) {
      if (!rows[a].empty() && *rows[a].rbegin() > rmax[a]) return false;  // cannot happen: the lattice lies inside the bound
      for (int r = 0; r <= rmax[a]; ++r) rows[a].insert(r);
    }
  }
  std::map<int, int> cidx[2];
  for (int a = 0; a < 2; ++a) {
    if ((int)rows[a].size() > thrl::kLut2MaxRows) return false;
    int c = 0;
    for (int row : rows[a]) {
      if (row < 0 || row > G.agent[a].states) return false;
      p->row_list[a][c] = (uint16_t)row;
      cidx[a][row] = c++;
    }
    p->NR[a] = c;
    const ThrlAgentSpec& s = G.agent[a];
    p->L[a] = s.min_memory > s.capacity ? 0 : (T < s.capacity ? T : s.capacity);
  }
  p->J = J;
  p->NS = NS;
  for (int j = 0; j < J; ++j) p->next_state[j] = (uint8_t)state_of[j];
  for (int s = 0; s < NS; ++s) {
    const auto& t = tuples[s];
    p->state_rows[s] = (uint32_t)cidx[0][t[0]] | ((uint32_t)cidx[0][t[1]] << 8) | ((uint32_t)cidx[1][t[2]] << 16) |
                       ((uint32_t)cidx[1][t[3]] << 24);
  }
  // shared-memory layout
  int o = 0;
  p->off_next = o;    o += align_up(2 * J, 16);
  p->off_rowlist = o; o += align_up(2 * (p->NR[0] + p->NR[1]), 16);
  p->off_lutlog = o;  o += J * 32;
  p->off_lutr = o;
  p->cta_bytes_lpc = o + J * 16;                                   // qtable_scan_lpc: [J][2] rewards
  o += align_up(J * 8, 16);
  p->off_aq = o;      o += align_up((A0 + A1) * 8, 16);            // qtable_scan_lut2: [J] prices, [A0 + A1] quantities
  p->cta_bytes = o;
  o = align_up((p->NR[0] + 2) * A0 * (int)elem, 16);
  p->off_tab1 = o;    o += align_up((p->NR[1] + 2) * A1 * (int)elem, 16);
  p->off_grow = o;    o += align_up(p->NR[0] + p->NR[1] + 4, 16);
  const int nstates = NS + 1 + (noisy ? T : 0);
  p->off_rows = o;    o += align_up(nstates * 4, 16);
  {  // lattice states, the initial state, the latest noise step's state; phase D's chunk scratch (+ read-ahead pad) reuses them
    const int gj = align_up((NS + 2) * 4, 16), scr = thrl::kLut2Chunk * 8 + 16;
    p->off_gj = o;    o += gj > scr ? gj : scr;
    p->off_scr = p->off_gj;
  }
  p->off_nt = o;      o += noisy ? align_up(T, 16) : 0;
  p->off_nrec = o;    o += noisy ? align_up(T * 8, 16) : 0;
  // the noise-free kernel derives the state before a step from the action record (nextS of the step before): no [T + 1]
  // state sequence, 112 B less per run at T = 100 (8,688 B at the C2 shape)
  p->off_seq = o;     o += noisy ? align_up(T + 1, 16) : 0;
  p->off_rec = o;     o += align_up(2 * T, 16);
  {  // phases A-B: pre[T] uint2; phases C-D: olds[T][2] -- disjoint lifetimes, one region
    const int pre = align_up(T * 8, 16), olds = align_up(2 * T * (int)elem, 16);
    p->off_old = o;   o += pre > olds ? pre : olds;
  }
  p->warp_bytes = o;
  const int w = (smem_optin - p->cta_bytes) / p->warp_bytes;
  if (w < 2) return false;
  int wmax = elem == 8 ? thrl::Lut2Warps<double>::kMax : thrl::Lut2Warps<float>::kMax;
  if (noisy && wmax > thrl::kLut2NoiseWarps) wmax = thrl::kLut2NoiseWarps;
  *warps = w > wmax ? wmax : w;
  return true;
}

template <typename QT>
int launch_lut2(thrl::Lut2Params& p, int warps, const DeviceInfo& dev, cudaStream_t stream) {
  int grid = dev.sms;
  g_last_wave = (long long)dev.sms * warps;
  const long long needed_ctas = (p.n_runs + warps - 1) / warps;
  if (needed_ctas < grid) {
    warps = (int)((p.n_runs + dev.sms - 1) / dev.sms);
    if (warps < 1) warps = 1;
    grid = (int)((p.n_runs + warps - 1) / warps);
  }
  const size_t smem = (size_t)p.cta_bytes + (size_t)warps * p.warp_bytes;
  const bool small = p.game.agent[0].actions <= 32 && p.game.agent[1].actions <= 32;
  auto kern = p.noisy ? (small ? thrl::qtable_scan_lut2<QT, true, true> : thrl::qtable_scan_lut2<QT, false, true>)
                      : (small ? thrl::qtable_scan_lut2<QT, true> : thrl::qtable_scan_lut2<QT, false>);
  CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  g_last_kernel = "lut2";
  kern<<<grid, warps * 32, smem, stream>>>(p);
  CUDA_TRY(cudaGetLastError());
  g_launches.fetch_add(1);
  return THRL_OK;
}

// ------------------------------------------------------------------------------------------------ LPC launch
template <typename QT, int GL>
int launch_lpc_gl(thrl::Lut2Params& p, const DeviceInfo& dev, cudaStream_t stream) {
  const ThrlGame& G = p.game;
  const int T = G.max_steps, esz = (int)sizeof(QT);
  thrl::LpcLayout lay;
  lay.cells_max = 0; lay.rows_max = 0;
  int Lmax = 1;
  for (int a = 0; a < 2; ++a) {
    const int cells = (p.NR[a] + 2) * G.agent[a].actions;
    if (cells > lay.cells_max) lay.cells_max = cells;
    if (p.NR[a] + 2 > lay.rows_max) lay.rows_max = p.NR[a] + 2;
    if (p.L[a] > Lmax) Lmax = p.L[a];
  }
  int o = 0;
  lay.off_tab = o;  o += align_up(lay.cells_max * GL * esz, 16);
  lay.off_old = o;  o += align_up(Lmax * GL * esz, 16);
  lay.off_rec = o;  o += align_up(T * GL * 4, 16);
  lay.off_pre = o;  o += align_up(T * GL, 16);
  lay.off_gj = o;   o += align_up((p.NS + 1) * GL * 4, 16);
  lay.off_rows = o; o += align_up((p.NS + 1) * GL * 2, 16);
  lay.off_grow = o; o += align_up(lay.rows_max * GL, 16);
  lay.off_eps = o;  o += align_up(GL * 8, 16);
  lay.off_xrow = o; o += align_up(2 * GL * 2, 16);
  lay.warp_bytes = o;
  int warps = (dev.smem_optin - p.cta_bytes_lpc) / lay.warp_bytes;
  if (warps < 1) return fail(THRL_ERR_UNSUPPORTED, "lpc: one warp group needs %d B of shared memory", lay.warp_bytes);
  if (warps > thrl::kLpcMaxWarps) warps = thrl::kLpcMaxWarps;
  const long long groups = (p.n_runs + GL / 2 - 1) / (GL / 2);
  int grid = dev.sms;
  if ((groups + warps - 1) / warps < grid) {
    warps = (int)((groups + dev.sms - 1) / dev.sms);
    if (warps < 1) warps = 1;
    grid = (int)((groups + warps - 1) / warps);
  }
  const size_t smem = (size_t)p.cta_bytes_lpc + (size_t)warps * lay.warp_bytes;
  // compile-time action count for the shapes the reference ships (example_config / configs2: 21 actions)
  const bool a21 = G.agent[0].actions == 21 && G.agent[1].actions == 21;
  auto kern = a21 ? thrl::qtable_scan_lpc<QT, GL, 21> : thrl::qtable_scan_lpc<QT, GL, 0>;
  CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  g_last_kernel = "lpc";
  g_last_wave = (long long)grid * warps * (GL / 2);
  kern<<<grid, warps * 32, smem, stream>>>(p, lay);
  CUDA_TRY(cudaGetLastError());
  g_launches.fetch_add(1);
  return THRL_OK;
}
template <typename QT>
int launch_lpc(thrl::Lut2Params& p, const DeviceInfo& dev, cudaStream_t stream) {
  const char* s = getenv("THRL_LPC_GL");
  const int gl = s ? atoi(s) : 8;
  switch (gl) {
    case 4: return launch_lpc_gl<QT, 4>(p, dev, stream);
    case 16: return launch_lpc_gl<QT, 16>(p, dev, stream);
    default: return launch_lpc_gl<QT, 8>(p, dev, stream);
  }
}

// ------------------------------------------------------------------------------------------------ mixed (MLP) launch
template <typename QT>
int launch_mixed(thrl::MixedParams& p, const DeviceInfo& dev, cudaStream_t stream) {
  const ThrlGame& G = p.game;
  const int n = G.n_agents, T = G.max_steps, Hp = p.Hp, esz = (int)sizeof(QT);
  int lut = 0, par = 0, pmax = 0, hmax = 0, amax = 0;
  for (int i = 0; i < n; ++i) {
    const ThrlAgentSpec& s = G.agent[i];
    lut += s.actions;
    p.par_off[i] = 0;
    if (s.kind == THRL_AGENT_QTABLE) continue;
    const int P = s.kind == THRL_AGENT_CAC ? 5 * s.hidden + 3 : 2 * s.hidden + s.actions * s.hidden + s.actions + (s.kind == THRL_AGENT_ACTORCRITIC ? s.hidden + 1 : 0);
    p.par_off[i] = par;
    par += align_up(P, 4);
    if (P > pmax) pmax = P;
    if (s.hidden > hmax) hmax = s.hidden;
    if (s.actions > amax) amax = s.actions;
  }
  p.lut_total = lut;
  p.cta_bytes = align_up(2 * lut * 8, 16);
  int o = 0;
  p.off_P = o;    o += align_up(Hp * 8, 16);
  p.off_newa = o; o += p.noisy ? align_up(T * 8, 16) : 0;
  p.off_hp = o;   o += align_up(n * 5 * 8, 16);
  p.off_old = o;  o += align_up(Hp * esz, 16);
  p.off_pre = o;  o += align_up(T * n * 4, 16);
  p.off_row = o;  o += align_up((Hp + 1) * 2, 16);
  p.off_act = o;  o += align_up(n * Hp, 16);
  p.off_par = o;  o += align_up(par * 4, 16);
  p.off_grad = o; o += align_up(pmax * 4, 16);
  p.off_h = o;    o += align_up((hmax + amax + 32) * 4, 16);
  p.warp_bytes = o;
  int warps = (dev.smem_optin - p.cta_bytes) / p.warp_bytes;
  if (warps < 1) return fail(THRL_ERR_UNSUPPORTED, "one run with its MLP agents needs %d B of shared memory (> %d B)", p.warp_bytes + p.cta_bytes, dev.smem_optin);
  if (warps > 16) warps = 16;
  int grid = dev.sms;
  {
    const long long slots = (long long)dev.sms * warps;
    const long long rounds = (p.n_runs + slots - 1) / slots;
    const long long per_round = (p.n_runs + rounds - 1) / rounds;
    warps = (int)((per_round + dev.sms - 1) / dev.sms);
    if (warps < 1) warps = 1;
    grid = (int)((per_round + warps - 1) / warps);
    if (grid > dev.sms) grid = dev.sms;
  }
  const size_t smem = (size_t)p.cta_bytes + (size_t)warps * p.warp_bytes;
  auto kern = thrl::qtable_scan_mixed<QT>;
  CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  g_last_kernel = "mixed";
  g_last_wave = (long long)grid * warps;
  kern<<<grid, warps * 32, smem, stream>>>(p);
  CUDA_TRY(cudaGetLastError());
  g_launches.fetch_add(1);
  return THRL_OK;
}

// ------------------------------------------------------------------------------------------------ lattice (pwl) launch
double h_scale_mlp(int k, int actions, double lo, double hi) {  // Reinforce.scale: k / actions * (hi - lo) + lo
  double d = (double)k / (double)actions;
  d = d * (hi - lo);
  return d + lo;
}
// builtin sum() of CPython >= 3.12 over scaled quantities whose first `lead` items are exact floats (thrl_device.cuh)
double h_py_sum(const double* aq, int n, int lead) {
  if (lead <= 2) {
    double q = 0.0;
    for (int i = 0; i < n; ++i) q = q + aq[i];
    return q;
  }
  double f = 0.0 + aq[0], c = 0.0;
  int i = 1;
  for (; i < lead; ++i) {
    const double x = aq[i], t = f + x;
    if (std::fabs(f) >= std::fabs(x)) { double d = f - t; d = d + x; c = c + d; }
    else { double d = x - t; d = d + f; c = c + d; }
    f = t;
  }
  if (c != 0.0 && std::isfinite(c)) f = f + c;
  for (; i < n; ++i) f = f + aq[i];
  return f;
}

static_assert(sizeof(thrl::PwlParams) < 32000, "kernel parameters are limited to 32,764 bytes");

// Fills p (lattice tables + layouts) when the game is one the lattice kernel plays: Reinforce / ActorCritic agents,
// optionally next to QTable agents of a regular game, on the noise-free demand curve, with few enough joint actions.
// Otherwise the order-exact kernel takes the game.  elem: bytes per Q-table cell.
bool plan_pwl(thrl::PwlParams* p, bool noisy, size_t elem, int smem_optin, int* warps) {
  const ThrlGame& G = p->game;
  const int n = G.n_agents, T = G.max_steps;
  if (noisy || n < 1) return false;
  long long J = 1;
  int lut = 0, Hmax = 1, Amax = 1, Pmax = 1, capmax = 0, nq = 0, lead = 0, rows_max = 0;
  bool leading = true;
  for (int i = 0; i < n; ++i) {
    const ThrlAgentSpec& s = G.agent[i];
    p->qidx[i] = -1;
    p->L[i] = 0;
    if (s.kind == THRL_AGENT_QTABLE) {
      if (!G.regular) return false;  // batches that span episodes: the order-exact kernel keeps the ring
      leading = false;
      p->qidx[i] = nq++;
      p->L[i] = s.min_memory > s.capacity ? 0 : (T < s.capacity ? T : s.capacity);
      if (s.states + 1 > rows_max) rows_max = s.states + 1;
    } else if (s.kind == THRL_AGENT_REINFORCE || s.kind == THRL_AGENT_ACTORCRITIC) {
      if (s.actions > 31 || s.hidden < 1) return false;
      if (s.entropy != 0.0) return false;  // the entropy regulariser is implemented by the interval-table and order-exact kernels
      if (leading) ++lead;
      const int P = 2 * s.hidden + s.actions * s.hidden + s.actions + (s.kind == THRL_AGENT_ACTORCRITIC ? s.hidden + 1 : 0);
      if (P > Pmax) Pmax = P;
      if (s.hidden > Hmax) Hmax = s.hidden;
      if (s.actions > Amax) Amax = s.actions;
      if (G.mlp_buffer_len[i] > capmax) capmax = G.mlp_buffer_len[i];
    } else {
      return false;
    }
    J *= s.actions;
    if (J > thrl::kPwlMaxJoint) return false;
    p->a_off[i] = lut;
    lut += s.actions;
  }
  p->J = (int)J;
  p->nq = nq;
  p->dwords = (rows_max + 31) / 32;
  p->lut_total = lut;
  p->jmul[n - 1] = 1;
  for (int i = n - 2; i >= 0; --i) p->jmul[i] = p->jmul[i + 1] * G.agent[i + 1].actions;
  const double ab = G.a / G.b;
  std::vector<float> fl((size_t)J);
  for (int j = 0; j < (int)J; ++j) {
    double aq[THRL_MAX_AGENTS];
    for (int i = 0; i < n; ++i) {
      const ThrlAgentSpec& s = G.agent[i];
      const int k = (j / p->jmul[i]) % s.actions;
      aq[i] = ab * (s.kind == THRL_AGENT_QTABLE ? h_scale(k, s.actions, s.action_lo, s.action_hi)
                                                : h_scale_mlp(k, s.actions, s.action_lo, s.action_hi));
    }
    const double Q = h_py_sum(aq, n, lead);
    const double pn = G.a - G.b * Q;
    const double price = pn > 0.0 ? pn : (pn != pn ? pn : 0.0);
    if (price != price) return false;
    p->priceJ[j] = price;
    fl[j] = (float)price;
  }
  std::vector<float> uniq(fl);
  std::sort(uniq.begin(), uniq.end());
  uniq.erase(std::unique(uniq.begin(), uniq.end()), uniq.end());
  const int NS = (int)uniq.size();
  if (NS > thrl::kPwlMaxLattice) return false;
  p->NS = NS;
  for (int x = 0; x < NS; ++x) p->slot_val[x] = uniq[x];
  for (int j = 0; j < (int)J; ++j)
    p->slot_of[j] = (uint16_t)(std::lower_bound(uniq.begin(), uniq.end(), fl[j]) - uniq.begin());
  const int NSX = NS + thrl::kPwlExtras;
  // shared memory
  int o = align_up(2 * lut * 8, 16);
  p->off_priceJ = o; o += align_up((int)J * 8, 16);
  p->off_rT = o;     o += align_up((int)J * n * 8, 16);
  p->off_rF = o;     o += align_up((int)J * n * 4, 16);
  p->off_slotof = o; o += align_up((int)J * 2, 16);
  p->off_urowJ = o;  o += align_up(nq * (int)J * 2, 16);
  p->cta_bytes = o;
  o = 0;
  p->off_sv = o;  o += align_up(NSX * 4, 16);
  int cdf = 0;
  for (int i = 0; i < n; ++i) {
    p->cdf_off[i] = cdf;
    p->val_off[i] = i * NSX;
    if (G.agent[i].kind != THRL_AGENT_QTABLE) cdf += NSX * G.agent[i].actions;
  }
  p->off_val = o; o += align_up(n * NSX * 4, 16);
  {  // the episode's draws; between episodes the same bytes stage kPwlTile hidden units of the forward sweep
    const int draws = T * n * 4, tile = thrl::kPwlTile * ((Amax + 1) * 4 + 12);
    p->off_pre = o; o += align_up(draws > tile ? draws : tile, 16);
  }
  p->off_ev = o;  o += align_up(Hmax * 2, 16);
  p->off_ord = o; o += align_up(Hmax * 2, 16);
  p->off_bkt = o; o += align_up((NS + 2) * 2, 16);
  p->off_hpw = o; o += align_up(n * 5 * 8, 16);
  p->off_jrec = o; o += nq ? align_up(T * 2, 16) : 0;
  p->off_oldv = o; o += nq ? align_up(T * (int)elem, 16) : 0;
  p->off_gq = o;   o += align_up(nq * NSX, 16);
  p->off_arow = o; o += align_up(nq * NSX * 2, 16);
  p->off_dirty = o; o += align_up(p->dwords * 4, 16);
  for (int i = 0; i < n; ++i) {
    p->off_tab[i] = o;
    if (G.agent[i].kind == THRL_AGENT_QTABLE) {
      const long long bytes = (long long)(G.agent[i].states + 1) * G.agent[i].row_stride * (long long)elem;
      if (bytes > smem_optin) return false;
      o += align_up((int)bytes, 16);
    }
  }
  // CDF LUT: in shared memory unless that leaves fewer than 8 runs resident per SM and the workspace (L2) placement more
  const int without = o, with = o + align_up(cdf * 4, 16);
  const int fit_with = (smem_optin - p->cta_bytes) / with, fit_without = (smem_optin - p->cta_bytes) / without;
  p->cdf_global = (fit_with < 8 && fit_without > fit_with) ? 1 : 0;
  p->off_cdf = o;
  p->warp_bytes = p->cdf_global ? without : with;
  // per-warp workspace in global memory
  long long w = 0;
  p->ws_acc = w;  w += align_up(NSX * (Amax + 2) * 8, 16);
  p->ws_pf = w;   w += align_up((NSX + 1) * (Amax + 1) * 16, 16);
  p->ws_p = w;    w += align_up((cdf > 0 ? cdf : 1) * 4, 16);
  p->ws_cdf = w;  w += p->cdf_global ? align_up(cdf * 4, 16) : 0;
  p->ws_grad = w; w += align_up(Pmax * 4, 16);
  p->ws_xs = w;   w += (long long)(capmax > 0 ? capmax : 1) * 16;
  p->ws_warp_bytes = (w + 255) / 256 * 256;
  const int fit = (smem_optin - p->cta_bytes) / p->warp_bytes;
  if (fit < 1) return false;
  *warps = fit > thrl::kPwlMaxWarps ? thrl::kPwlMaxWarps : fit;
  if (const char* f = getenv("THRL_PWL_WARPS"))
    if (atoi(f) >= 1 && atoi(f) < *warps) *warps = atoi(f);
  return true;
}

// The library's own stream-ordered pool for the lattice kernel's workspace (one per device).  It keeps what it has been given
// instead of returning it to the driver at every synchronisation (release threshold), so steady-state calls allocate nothing.
cudaMemPool_t pwl_pool(int device, bool create) {
  static cudaMemPool_t pools[64] = {};
  static std::mutex pool_mu;
  std::lock_guard<std::mutex> lock(pool_mu);
  if (!pools[device] && create) {
    cudaMemPoolProps props = {};
    props.allocType = cudaMemAllocationTypePinned;
    props.location.type = cudaMemLocationTypeDevice;
    props.location.id = device;
    if (cudaMemPoolCreate(&pools[device], &props) != cudaSuccess) { pools[device] = nullptr; return nullptr; }
    unsigned long long keep = ~0ull;
    cudaMemPoolSetAttribute(pools[device], cudaMemPoolAttrReleaseThreshold, &keep);
  }
  return pools[device];
}

int launch_pwl(thrl::PwlParams& p, int warps, bool f64, const DeviceInfo& dev, cudaStream_t stream) {
  // A call that needs several rounds of the persistent grid is launched round by round (same stream, runs [lo, hi) each):
  // warps that start a round together stay in step through its episodes and updates, which a single launch of seven rounds
  // loses after the first one (C5: 4.15e9 against 3.0-4.0e9 agent-steps/s; runs are independent, so the result is the same).
  const long long slots = (long long)dev.sms * warps;
  const long long total = p.n_runs;
  // stream-ordered scratch from the library's own pool
  int device = 0;
  CUDA_TRY(cudaGetDevice(&device));
  if (device < 0 || device >= 64) return fail(THRL_ERR_BAD_ARGS, "device index %d", device);
  cudaMemPool_t pool = pwl_pool(device, true);
  if (!pool) return fail(THRL_ERR_CUDA, "cudaMemPoolCreate failed: %s", cudaGetErrorString(cudaGetLastError()));
  void* ws = nullptr;
  CUDA_TRY(cudaMallocFromPoolAsync(&ws, (size_t)dev.sms * warps * (size_t)p.ws_warp_bytes, pool, stream));
  p.ws = (unsigned char*)ws;
  const bool two = p.game.n_agents == 2, g = p.cdf_global != 0;
  void (*kern)(thrl::PwlParams);
  if (p.nq == 0) {  // no tables: the table type does not enter
    kern = two ? (g ? thrl::mlp_scan_pwl<float, 2, false, true> : thrl::mlp_scan_pwl<float, 2, false, false>)
               : (g ? thrl::mlp_scan_pwl<float, 0, false, true> : thrl::mlp_scan_pwl<float, 0, false, false>);
  } else if (f64) {
    kern = two ? (g ? thrl::mlp_scan_pwl<double, 2, true, true> : thrl::mlp_scan_pwl<double, 2, true, false>)
               : (g ? thrl::mlp_scan_pwl<double, 0, true, true> : thrl::mlp_scan_pwl<double, 0, true, false>);
  } else {
    kern = two ? (g ? thrl::mlp_scan_pwl<float, 2, true, true> : thrl::mlp_scan_pwl<float, 2, true, false>)
               : (g ? thrl::mlp_scan_pwl<float, 0, true, true> : thrl::mlp_scan_pwl<float, 0, true, false>);
  }
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)((size_t)p.cta_bytes + (size_t)warps * p.warp_bytes));
  g_last_kernel = "pwl";
  g_last_wave = slots;
  for (long long lo = 0; lo < total && e == cudaSuccess; lo += slots) {
    const long long n = total - lo < slots ? total - lo : slots;
    int w = (int)((n + dev.sms - 1) / dev.sms);
    if (w < 1) w = 1;
    int grid = (int)((n + w - 1) / w);
    if (grid > dev.sms) grid = dev.sms;
    p.run_lo = lo;
    p.n_runs = lo + n;
    kern<<<grid, w * 32, (size_t)p.cta_bytes + (size_t)w * p.warp_bytes, stream>>>(p);
    e = cudaGetLastError();
    g_launches.fetch_add(1);
  }
  p.n_runs = total;
  cudaFreeAsync(ws, stream);
  CUDA_TRY(e);
  return THRL_OK;
}

// ------------------------------------------------------------------------------------------------ continuous-state MLP (pwc) launch
// Fills p (layouts) when the interval-table kernel plays the game: at least one MLP agent, every MLP agent with at most
// kPwcMaxHidden hidden units and at most 32 head columns.  It takes what the lattice kernel cannot: demand noise, CAC agents,
// QTable agents whose batches span episodes.
bool plan_pwc(thrl::PwcParams* p, bool noisy, size_t elem, int smem_optin, int* warps) {
  const ThrlGame& G = p->game;
  const int n = G.n_agents, T = G.max_steps;
  p->noisy = noisy ? 1 : 0;
  p->Hp = (G.ring_len > 0 ? G.ring_len : 1) + 1;
  const int Hp = p->Hp;
  int lut = 0, Hmax = 0, ncpmax = 0, Pmax = 1, capmax = 0, nm = 0;
  long long w = 0;
  int o = 0;
  p->off_P = o;    o += align_up(Hp * 8, 16);
  p->off_newa = o; o += noisy ? align_up(T * 8, 16) : 0;
  p->off_hp = o;   o += align_up(n * 5 * 8, 16);
  p->off_old = o;  o += align_up(Hp * (int)elem, 16);
  p->off_pre = o;  o += align_up(T * n * 4, 16);
  p->off_zf = o;   o += align_up(T * n * 4, 16);
  p->off_row = o;  o += align_up((Hp + 1) * 2, 16);
  p->off_act = o;  o += align_up(n * Hp, 16);
  for (int i = 0; i < n; ++i) {
    const ThrlAgentSpec& s = G.agent[i];
    lut += s.actions;
    p->off_th[i] = 0; p->ncp[i] = 0; p->ws_tab[i] = 0; p->ws_ord[i] = 0;
    if (s.kind == THRL_AGENT_QTABLE) continue;
    const int H = s.hidden;
    const int nc = s.kind == THRL_AGENT_CAC ? 3 : s.actions + (s.kind == THRL_AGENT_ACTORCRITIC ? 1 : 0);
    if (H < 1 || H > thrl::kPwcMaxHidden || nc > 32 || (s.kind != THRL_AGENT_CAC && s.actions < 1)) return false;
    ++nm;
    const int P = s.kind == THRL_AGENT_CAC ? 5 * H + 3 : 2 * H + s.actions * H + s.actions + (s.kind == THRL_AGENT_ACTORCRITIC ? H + 1 : 0);
    p->ncp[i] = align_up(nc, 2);
    p->off_th[i] = o; o += (((H + 31) / 32) * 32 + 32) * 4;  // ranked thresholds padded to whole blocks, then the 32 block maxima
    p->ws_tab[i] = w; w += align_up((H + 1) * p->ncp[i] * 16, 256);
    p->ws_ord[i] = w; w += align_up(H * 2, 256);
    if (H > Hmax) Hmax = H;
    if (p->ncp[i] > ncpmax) ncpmax = p->ncp[i];
    if (P > Pmax) Pmax = P;
    if (G.mlp_buffer_len[i] > capmax) capmax = G.mlp_buffer_len[i];
  }
  if (nm == 0) return false;
  p->lut_total = lut;
  p->cta_bytes = align_up(2 * lut * 8, 16);
  p->off_hist = o; o += align_up((Hmax + 3) * 4, 16);
  p->warp_bytes = o;
  p->ws_bkt = w;  w += align_up((Hmax + 2) * ncpmax * 16, 256);
  p->ws_grad = w; w += align_up(Pmax * 4, 256);
  p->ws_xs = w;   w += align_up((capmax > 0 ? capmax : 1) * 16, 256);
  p->ws_xe = w;   w += align_up((capmax > 0 ? capmax : 1) * 4, 256);
  p->ws_evs = w;  w += (long long)(capmax > 0 ? capmax : 1) * 8;
  p->ws_warp_bytes = (w + 255) / 256 * 256;
  const int fit = (smem_optin - p->cta_bytes) / p->warp_bytes;
  if (fit < 1) return false;
  // 16 warps x 128 registers.  (24 warps under __launch_bounds__(768, 1) = 80 registers measured 8 % slower: 300 B of spills.)
  int cap = thrl::kPwcMaxWarps;
  if (const char* f = getenv("THRL_PWC_WARPS")) cap = atoi(f) < 1 ? 1 : (atoi(f) > thrl::kPwcMaxWarps ? thrl::kPwcMaxWarps : atoi(f));
  *warps = fit > cap ? cap : fit;
  return true;
}

template <typename QT>
int launch_pwc(thrl::PwcParams& p, int warps, const DeviceInfo& dev, cudaStream_t stream) {
  int grid = dev.sms;
  {
    const long long slots = (long long)dev.sms * warps;
    const long long rounds = (p.n_runs + slots - 1) / slots;
    const long long per_round = (p.n_runs + rounds - 1) / rounds;
    warps = (int)((per_round + dev.sms - 1) / dev.sms);
    if (warps < 1) warps = 1;
    grid = (int)((per_round + warps - 1) / warps);
    if (grid > dev.sms) grid = dev.sms;
  }
  const size_t smem = (size_t)p.cta_bytes + (size_t)warps * p.warp_bytes;
  int device = 0;
  CUDA_TRY(cudaGetDevice(&device));
  if (device < 0 || device >= 64) return fail(THRL_ERR_BAD_ARGS, "device index %d", device);
  cudaMemPool_t pool = pwl_pool(device, true);
  if (!pool) return fail(THRL_ERR_CUDA, "cudaMemPoolCreate failed: %s", cudaGetErrorString(cudaGetLastError()));
  void* ws = nullptr;
  CUDA_TRY(cudaMallocFromPoolAsync(&ws, (size_t)grid * warps * (size_t)p.ws_warp_bytes, pool, stream));
  p.ws = (unsigned char*)ws;
  const ThrlGame& G = p.game;
  const bool two = G.n_agents == 2 && (G.agent[0].kind == THRL_AGENT_REINFORCE || G.agent[0].kind == THRL_AGENT_ACTORCRITIC) &&
                   (G.agent[1].kind == THRL_AGENT_REINFORCE || G.agent[1].kind == THRL_AGENT_ACTORCRITIC);
  auto kern = two ? thrl::mlp_scan_pwc<QT, true> : thrl::mlp_scan_pwc<QT, false>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e == cudaSuccess) {
    g_last_kernel = "pwc";
    g_last_wave = (long long)grid * warps;
    kern<<<grid, warps * 32, smem, stream>>>(p);
    e = cudaGetLastError();
  }
  cudaFreeAsync(ws, stream);
  CUDA_TRY(e);
  g_launches.fetch_add(1);
  return THRL_OK;
}

// Plans (structure tables + shared-memory layouts) are functions of the laid-out game, the cell size and the noise flag only:
// they are built once and copied per call (train_one's small chunks and the host pipeline launch the same game many times).
template <typename P>
struct PlanCache {
  struct Entry { ThrlGame g; int elem, noisy, smem; bool ok; int warps; std::unique_ptr<P> plan; };
  std::vector<Entry> entries;
  std::mutex mu;
  // Returns whether the kernel applies; on true *out holds the plan (pointers and run counts zero) and *warps its residency.
  template <typename F>
  bool get(const ThrlGame& G, int elem, int noisy, int smem, P* out, int* warps, F build) {
    std::lock_guard<std::mutex> lock(mu);
    for (auto& e : entries)
      if (e.elem == elem && e.noisy == noisy && e.smem == smem && memcmp(&e.g, &G, sizeof(G)) == 0) {
        if (e.ok) { *out = *e.plan; *warps = e.warps; }
        return e.ok;
      }
    Entry e{G, elem, noisy, smem, false, 0, std::unique_ptr<P>(new P())};
    memset(e.plan.get(), 0, sizeof(P));
    e.plan->game = G;
    e.ok = build(e.plan.get(), &e.warps);
    if (e.ok) { *out = *e.plan; *warps = e.warps; }
    const bool ok = e.ok;
    if (entries.size() >= 16) entries.erase(entries.begin());
    entries.push_back(std::move(e));
    return ok;
  }
};
PlanCache<thrl::Lut2Params> g_lut2_plans;
PlanCache<thrl::PwlParams> g_pwl_plans;
PlanCache<thrl::PwcParams> g_pwc_plans;

int check_args(const ThrlScanArgs* a) {
  if (!a || !a->game) return fail(THRL_ERR_BAD_ARGS, "args/game is NULL");
  if (a->n_runs < 0 || a->epoch_end < a->epoch_begin) return fail(THRL_ERR_BAD_ARGS, "negative run or epoch count");
  if (a->table_dtype != THRL_F32 && a->table_dtype != THRL_F64) return fail(THRL_ERR_BAD_ARGS, "table_dtype=%d", a->table_dtype);
  if (a->rng_mode < THRL_RNG_PHILOX || a->rng_mode > THRL_RNG_REPLAY_ACTIONS) return fail(THRL_ERR_BAD_ARGS, "rng_mode=%d", a->rng_mode);
  if (!a->eps || !a->price) return fail(THRL_ERR_BAD_ARGS, "eps / price must not be NULL");
  if (a->rng_mode != THRL_RNG_PHILOX && !a->replay_ra) return fail(THRL_ERR_BAD_ARGS, "replay mode without replay_ra");
  if (a->rng_mode == THRL_RNG_REPLAY_DRAWS && !a->replay_u) return fail(THRL_ERR_BAD_ARGS, "REPLAY_DRAWS without replay_u");
  bool has_mlp = false;
  for (int i = 0; i < a->game->n_agents && i < THRL_MAX_AGENTS; ++i) has_mlp |= a->game->agent[i].kind != THRL_AGENT_QTABLE;
  if (has_mlp && !a->mlp) return fail(THRL_ERR_BAD_ARGS, "the game has MLP agents but args->mlp is NULL");
  if (a->n_log_runs < 0 || a->n_log_runs > a->n_runs) return fail(THRL_ERR_BAD_ARGS, "n_log_runs=%lld outside 0..n_runs", (long long)a->n_log_runs);
  // Philox counters carry the global run id in one 32-bit word (thrl_device.cuh): ids beyond 2^32 would alias streams
  if (a->run_id0 < 0 || a->run_id0 + a->n_runs > (1LL << 32))
    return fail(THRL_ERR_BAD_ARGS, "global run ids [%lld, %lld) leave the 32-bit range of the Philox counter word", (long long)a->run_id0,
                (long long)(a->run_id0 + a->n_runs));
  return THRL_OK;
}

// Checks that need the laid-out game: the carried ring of non-regular games, and the range of the fixed-point statistics.
int check_args_game(const ThrlScanArgs* a, const ThrlGame& G) {
  if (!G.regular && !a->ring)
    return fail(THRL_ERR_BAD_ARGS, "the game is not regular (an agent's min_memory exceeds max_steps, so transitions are pending at "
                                   "epoch boundaries): args->ring is required (thrl_ring_bytes per run, zero-filled = empty buffers)");
  if (a->stats) {
    // sums over the call's runs of r * 2^32 and r^2 * 2^24 in int64 (accumulated across calls by the caller: leave 2 bits).
    // |per-epoch mean reward| <= price * quantity <= a * (a/b) * max|action|, |mean action| <= max|action|.
    double xmax = 0.0;
    for (int i = 0; i < G.n_agents; ++i) {
      const double m = std::fmax(std::fabs(G.agent[i].action_lo), std::fabs(G.agent[i].action_hi));
      if (m > xmax) xmax = m;
    }
    const double rmax = std::fabs(G.a) * std::fabs(G.a / G.b) * xmax, big = std::fmax(rmax, xmax);
    const double lim = 2305843009213693952.0;  // 2^61
    if (!(big * THRL_STATS_SCALE_SUM * (double)a->n_runs < lim) || !(big * big * THRL_STATS_SCALE_SQ * (double)a->n_runs < lim))
      return fail(THRL_ERR_UNSUPPORTED, "stats: %lld runs of rewards up to %g would overflow the fixed-point sums (THRL_STATS_SCALE_*); "
                                        "split the call or pass stats = NULL", (long long)a->n_runs, rmax);
  }
  return THRL_OK;
}

}  // namespace

extern "C" {

int thrl_abi_version(void) { return THRL_ABI_VERSION; }
const char* thrl_last_error(void) { return g_err; }
int64_t thrl_launch_count(void) { return (int64_t)g_launches.load(); }
const char* thrl_last_kernel(void) { return g_last_kernel; }
int64_t thrl_last_wave_runs(void) { return g_last_wave; }

int thrl_game_layout(ThrlGame* game) { return validate_layout(game); }

int64_t thrl_ring_bytes(const ThrlGame* game) {
  ThrlGame g = *game;
  if (validate_layout(&g) != THRL_OK) return -1;
  return ring_bytes(&g);
}

int thrl_qtable_scan(const ThrlScanArgs* a, void* stream_) {
  int rc = check_args(a);
  if (rc) return rc;
  thrl::ScanParams p;
  memset(&p, 0, sizeof(p));
  p.game = *a->game;
  rc = validate_layout(&p.game);
  if (rc) return rc;
  if (p.game.run_stride > 0 && !a->q) return fail(THRL_ERR_BAD_ARGS, "q must not be NULL (the game has Q-tables)");
  rc = check_args_game(a, p.game);
  if (rc) return rc;
  if (a->n_runs == 0 || a->epoch_end == a->epoch_begin) return THRL_OK;
  DeviceInfo dev;
  rc = device_info(&dev);
  if (rc) return rc;
  p.n_runs = a->n_runs;
  p.run_id0 = a->run_id0;
  p.epoch_begin = a->epoch_begin;
  p.E = a->epoch_end - a->epoch_begin;
  p.rng_mode = a->rng_mode;
  p.k0 = (uint32_t)a->seed;
  p.k1 = (uint32_t)(a->seed >> 32);
  p.q = a->q; p.counter = a->counter; p.eps = a->eps; p.price = a->price; p.hp = a->hp;
  p.ring = (unsigned char*)a->ring;
  p.ring_bytes = ring_bytes(&p.game);
  p.replay_u = a->replay_u; p.replay_ra = a->replay_ra; p.replay_new_a = a->replay_new_a;
  p.rewards_log = a->rewards_log; p.actions_log = a->actions_log; p.n_log_runs = a->n_log_runs;
  p.stats = (long long*)a->stats;
  p.trace_actions = a->trace_actions; p.trace_rewards = a->trace_rewards; p.trace_prices = a->trace_prices;
  p.Hp = (p.game.ring_len > 0 ? p.game.ring_len : 1) + 1;
  p.noisy = (a->rng_mode == THRL_RNG_PHILOX) ? (p.game.noise_prob > 0.0) : (a->replay_new_a != nullptr);
  cudaStream_t stream = (cudaStream_t)stream_;
  if (p.game.mlp_stride > 0) {  // games with MLP agents
    const char* forced = getenv("THRL_KERNEL");
    const bool want_mixed = forced && strcmp(forced, "mixed") == 0, want_pwc = forced && strcmp(forced, "pwc") == 0;
    if (!want_mixed && !want_pwc) {  // lattice kernel where it applies (thrl_scan_pwl.cuh)
      thrl::PwlParams* w = new thrl::PwlParams();
      std::unique_ptr<thrl::PwlParams> hold_w(w);
      int warps = 0;
      const int elem = a->table_dtype == THRL_F64 ? 8 : 4;
      if (g_pwl_plans.get(p.game, elem, p.noisy, dev.smem_optin, w, &warps, [&](thrl::PwlParams* q, int* wq) {
            return plan_pwl(q, p.noisy != 0, (size_t)elem, dev.smem_optin, wq);
          })) {
        w->n_runs = p.n_runs; w->run_id0 = p.run_id0; w->epoch_begin = p.epoch_begin; w->E = p.E; w->rng_mode = p.rng_mode;
        w->k0 = p.k0; w->k1 = p.k1;
        w->price = p.price; w->replay_ra = p.replay_ra; w->replay_u = p.replay_u;
        w->q = p.q; w->counter = p.counter; w->eps = p.eps; w->hp = p.hp;
        w->rewards_log = p.rewards_log; w->actions_log = p.actions_log; w->n_log_runs = p.n_log_runs; w->stats = p.stats;
        w->trace_actions = p.trace_actions; w->trace_rewards = p.trace_rewards; w->trace_prices = p.trace_prices;
        w->mlp = a->mlp;
        return launch_pwl(*w, warps, a->table_dtype == THRL_F64, dev, stream);
      }
    }
    if (!want_mixed) {  // continuous prices (demand noise, CAC, pending QTable batches): interval-table kernel (thrl_scan_pwc.cuh)
      thrl::PwcParams* w = new thrl::PwcParams();
      std::unique_ptr<thrl::PwcParams> hold_w(w);
      int warps = 0;
      const int elem = a->table_dtype == THRL_F64 ? 8 : 4;
      if (g_pwc_plans.get(p.game, elem, p.noisy, dev.smem_optin, w, &warps, [&](thrl::PwcParams* q, int* wq) {
            return plan_pwc(q, p.noisy != 0, (size_t)elem, dev.smem_optin, wq);
          })) {
        w->n_runs = p.n_runs; w->run_id0 = p.run_id0; w->epoch_begin = p.epoch_begin; w->E = p.E; w->rng_mode = p.rng_mode;
        w->k0 = p.k0; w->k1 = p.k1;
        w->q = p.q; w->counter = p.counter; w->eps = p.eps; w->price = p.price; w->hp = p.hp;
        w->replay_u = p.replay_u; w->replay_ra = p.replay_ra; w->replay_new_a = p.replay_new_a;
        w->rewards_log = p.rewards_log; w->actions_log = p.actions_log; w->n_log_runs = p.n_log_runs; w->stats = p.stats;
        w->trace_actions = p.trace_actions; w->trace_rewards = p.trace_rewards; w->trace_prices = p.trace_prices;
        w->mlp = a->mlp; w->ring = p.ring; w->ring_bytes = p.ring_bytes;
        return a->table_dtype == THRL_F64 ? launch_pwc<double>(*w, warps, dev, stream) : launch_pwc<float>(*w, warps, dev, stream);
      }
    }
    thrl::MixedParams* m = new thrl::MixedParams();
    std::unique_ptr<thrl::MixedParams> hold(m);
    m->game = p.game;
    m->n_runs = p.n_runs; m->run_id0 = p.run_id0; m->epoch_begin = p.epoch_begin; m->E = p.E; m->rng_mode = p.rng_mode;
    m->k0 = p.k0; m->k1 = p.k1;
    m->q = p.q; m->counter = p.counter; m->eps = p.eps; m->price = p.price; m->hp = p.hp;
    m->replay_u = p.replay_u; m->replay_ra = p.replay_ra; m->replay_new_a = p.replay_new_a;
    m->rewards_log = p.rewards_log; m->actions_log = p.actions_log; m->n_log_runs = p.n_log_runs; m->stats = p.stats;
    m->trace_actions = p.trace_actions; m->trace_rewards = p.trace_rewards; m->trace_prices = p.trace_prices;
    m->mlp = a->mlp; m->Hp = p.Hp; m->noisy = p.noisy; m->ring = p.ring; m->ring_bytes = p.ring_bytes;
    return a->table_dtype == THRL_F64 ? launch_mixed<double>(*m, dev, stream) : launch_mixed<float>(*m, dev, stream);
  }
  // Kernel choice.  THRL_KERNEL=generic forces the general kernel, lut2 / lpc pick one of the two specialised kernels
  // where they apply (tests exercise all three); default: see below.
  const char* force = getenv("THRL_KERNEL");
  const bool want_generic = force && strcmp(force, "generic") == 0;
  if (!want_generic) {
    thrl::Lut2Params* l = new thrl::Lut2Params();
    std::unique_ptr<thrl::Lut2Params> hold(l);
    int warps = 0;
    const int elem = a->table_dtype == THRL_F64 ? 8 : 4;
    if (g_lut2_plans.get(p.game, elem, p.noisy, dev.smem_optin, l, &warps, [&](thrl::Lut2Params* q, int* wq) {
          return plan_lut2(q, p.noisy != 0, (size_t)elem, dev.smem_optin, wq);
        })) {
      l->n_runs = p.n_runs; l->run_id0 = p.run_id0; l->epoch_begin = p.epoch_begin; l->E = p.E; l->rng_mode = p.rng_mode;
      l->k0 = p.k0; l->k1 = p.k1;
      l->q = p.q; l->counter = p.counter; l->eps = p.eps; l->price = p.price; l->hp = p.hp;
      l->replay_u = p.replay_u; l->replay_ra = p.replay_ra; l->replay_new_a = p.replay_new_a;
      l->rewards_log = p.rewards_log; l->actions_log = p.actions_log; l->n_log_runs = p.n_log_runs; l->stats = p.stats;
      l->trace_actions = p.trace_actions; l->trace_rewards = p.trace_rewards; l->trace_prices = p.trace_prices;
      if (force && strcmp(force, "lpc") == 0 && !l->noisy)  // the lane-per-chain variant is noise-free only
        return a->table_dtype == THRL_F64 ? launch_lpc<double>(*l, dev, stream) : launch_lpc<float>(*l, dev, stream);
      return a->table_dtype == THRL_F64 ? launch_lut2<double>(*l, warps, dev, stream) : launch_lut2<float>(*l, warps, dev, stream);
    }
  }
  if (!want_generic) {  // tables that stay in HBM: gather / on-chip walk kernel (thrl_scan_hbm.cuh)
    thrl::HbmParams h;
    memset(&h, 0, sizeof(h));
    h.game = p.game;
    h.n_runs = p.n_runs;
    h.E = p.E;
    h.noisy = p.noisy;
    int warps = 0;
    if (plan_hbm(&h, a->table_dtype == THRL_F64 ? 8 : 4, dev, &warps)) {
      h.run_id0 = p.run_id0; h.epoch_begin = p.epoch_begin; h.E = p.E; h.rng_mode = p.rng_mode;
      h.k0 = p.k0; h.k1 = p.k1;
      h.q = p.q; h.counter = p.counter; h.eps = p.eps; h.price = p.price; h.hp = p.hp;
      h.replay_u = p.replay_u; h.replay_ra = p.replay_ra; h.replay_new_a = p.replay_new_a;
      h.rewards_log = p.rewards_log; h.actions_log = p.actions_log; h.n_log_runs = p.n_log_runs; h.stats = p.stats;
      h.trace_actions = p.trace_actions; h.trace_rewards = p.trace_rewards; h.trace_prices = p.trace_prices;
      if (((uintptr_t)h.q & 15u) != 0) return fail(THRL_ERR_BAD_ARGS, "q must be 16-byte aligned (padded slab layout, include/thrl.h)");
      return a->table_dtype == THRL_F64 ? launch_hbm<double>(h, warps, dev, stream) : launch_hbm<float>(h, warps, dev, stream);
    }
  }
  return a->table_dtype == THRL_F64 ? launch_generic<double>(p, dev, stream) : launch_generic<float>(p, dev, stream);
}

int thrl_qtable_init(const ThrlGame* game, int64_t n_runs, int64_t run_id0, uint64_t seed, int32_t table_dtype,
                     const double* hp, const double* eps0, void* q, uint32_t* counter, double* eps, double* price,
                     void* stream) {
  return thrl_game_init(game, n_runs, run_id0, seed, table_dtype, hp, eps0, q, counter, eps, price, nullptr, stream);
}

int thrl_game_init(const ThrlGame* game, int64_t n_runs, int64_t run_id0, uint64_t seed, int32_t table_dtype,
                   const double* hp, const double* eps0, void* q, uint32_t* counter, double* eps, double* price, float* mlp,
                   void* stream) {
  if (!game || !eps0 || !eps || !price) return fail(THRL_ERR_BAD_ARGS, "thrl_game_init: NULL argument");
  if (table_dtype != THRL_F32 && table_dtype != THRL_F64) return fail(THRL_ERR_BAD_ARGS, "table_dtype=%d", table_dtype);
  thrl::InitParams p;
  memset(&p, 0, sizeof(p));
  p.game = *game;
  int rc = validate_layout(&p.game);
  if (rc) return rc;
  if (n_runs <= 0) return THRL_OK;
  DeviceInfo dev;
  rc = device_info(&dev);
  if (rc) return rc;
  p.n_runs = n_runs; p.run_id0 = run_id0;
  p.k0 = (uint32_t)seed; p.k1 = (uint32_t)(seed >> 32);
  p.f64 = table_dtype == THRL_F64;
  p.hp = hp;
  for (int i = 0; i < p.game.n_agents; ++i) p.eps0[i] = eps0[i];
  p.q = q; p.counter = counter; p.eps = eps; p.price = price; p.mlp = mlp;
  if (p.game.mlp_stride > 0 && !mlp) return fail(THRL_ERR_BAD_ARGS, "the game has MLP agents but mlp is NULL");
  if (p.game.run_stride > 0 && !q) return fail(THRL_ERR_BAD_ARGS, "q must not be NULL (the game has Q-tables)");
  long long max_cells = 0;
  for (int i = 0; i < p.game.n_agents; ++i) {
    const ThrlAgentSpec& sa = p.game.agent[i];
    const long long c = sa.kind == THRL_AGENT_QTABLE ? (long long)(sa.states + 1) * sa.actions : 2 * (3LL * (3 * sa.hidden + sa.actions * sa.hidden + sa.actions + 1) + 4 + 4LL * p.game.mlp_buffer_len[i]);
    if (c > max_cells) max_cells = c;
  }
  dim3 grid((unsigned)((max_cells / 2 + 255) / 256), (unsigned)(n_runs < 65535 ? n_runs : 65535));
  if (grid.x < 1) grid.x = 1;
  if (grid.x > 64) grid.x = 64;
  thrl::qtable_init<<<grid, 256, 0, (cudaStream_t)stream>>>(p);
  CUDA_TRY(cudaGetLastError());
  g_launches.fetch_add(1);
  return THRL_OK;
}

int thrl_greedy_eval(const ThrlGame* game, int64_t n_runs, int32_t table_dtype, const void* q, int32_t iters,
                     const double* price0, double* rewards, double* actions, void* stream) {
  return thrl_greedy_eval_mlp(game, n_runs, table_dtype, q, nullptr, iters, price0, rewards, actions, stream);
}

int thrl_greedy_eval_mlp(const ThrlGame* game, int64_t n_runs, int32_t table_dtype, const void* q, const float* mlp,
                         int32_t iters, const double* price0, double* rewards, double* actions, void* stream) {
  return thrl_greedy_eval_noise(game, n_runs, table_dtype, q, mlp, iters, price0, nullptr, rewards, actions, stream);
}

int thrl_greedy_eval_noise(const ThrlGame* game, int64_t n_runs, int32_t table_dtype, const void* q, const float* mlp,
                           int32_t iters, const double* price0, const double* new_a, double* rewards, double* actions, void* stream) {
  if (!game || !price0 || !rewards || !actions) return fail(THRL_ERR_BAD_ARGS, "thrl_greedy_eval: NULL argument");
  if (table_dtype != THRL_F32 && table_dtype != THRL_F64) return fail(THRL_ERR_BAD_ARGS, "table_dtype=%d", table_dtype);
  ThrlGame G = *game;
  int rc = validate_layout(&G);
  if (rc) return rc;
  if (G.run_stride > 0 && !q) return fail(THRL_ERR_BAD_ARGS, "q must not be NULL (the game has Q-tables)");
  if (G.mlp_stride > 0 && !mlp) return fail(THRL_ERR_BAD_ARGS, "the game has MLP agents but mlp is NULL");
  // utils.play_game steps the environment, which perturbs the demand intercept when noise_prob > 0 (environments.py:28-31);
  // without the intercept stream a noisy game is refused instead of being played without noise
  if (G.noise_prob > 0.0 && !new_a)
    return fail(THRL_ERR_UNSUPPORTED, "thrl_greedy_eval: noise_prob=%g > 0 needs the demand intercepts of the steps "
                                      "(thrl_greedy_eval_noise, new_a)", G.noise_prob);
  if (n_runs <= 0 || iters <= 0) return THRL_OK;
  DeviceInfo dev;
  rc = device_info(&dev);
  if (rc) return rc;
  long long blocks = (n_runs + 7) / 8;
  if (blocks > dev.sms * 8) blocks = dev.sms * 8;
  if (G.mlp_stride == 0) {
    thrl::EvalParams p;
    memset(&p, 0, sizeof(p));
    p.game = G;
    p.n_runs = n_runs; p.iters = iters; p.q = q; p.price0 = price0; p.new_a = new_a; p.rewards = rewards; p.actions = actions;
    if (table_dtype == THRL_F64) thrl::greedy_eval<double><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(p);
    else thrl::greedy_eval<float><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(p);
  } else {
    thrl::EvalMixedParams* p = new thrl::EvalMixedParams();
    std::unique_ptr<thrl::EvalMixedParams> hold(p);
    memset(p, 0, sizeof(*p));
    p->game = G;
    p->n_runs = n_runs; p->iters = iters; p->q = q; p->mlp = mlp; p->price0 = price0; p->new_a = new_a; p->rewards = rewards; p->actions = actions;
    int par = 0, hmax = 0, amax = 0;
    for (int i = 0; i < G.n_agents; ++i) {
      const ThrlAgentSpec& s = G.agent[i];
      if (s.kind == THRL_AGENT_QTABLE) continue;
      const int P = s.kind == THRL_AGENT_CAC ? 5 * s.hidden + 3 : 2 * s.hidden + s.actions * s.hidden + s.actions + (s.kind == THRL_AGENT_ACTORCRITIC ? s.hidden + 1 : 0);
      p->par_off[i] = par;
      par += align_up(P, 4);
      if (s.hidden > hmax) hmax = s.hidden;
      if (s.actions > amax) amax = s.actions;
    }
    p->off_par = 0;
    p->off_h = align_up(par * 4, 16);
    p->warp_bytes = p->off_h + align_up((hmax + amax + 32) * 4, 16);
    int warps = dev.smem_optin / p->warp_bytes;
    if (warps < 1) return fail(THRL_ERR_UNSUPPORTED, "one run's MLP agents need %d B of shared memory", p->warp_bytes);
    if (warps > 8) warps = 8;
    const size_t smem = (size_t)warps * p->warp_bytes;
    blocks = (n_runs + warps - 1) / warps;
    if (blocks > dev.sms) blocks = dev.sms;
    auto kern = table_dtype == THRL_F64 ? thrl::greedy_eval_mixed<double> : thrl::greedy_eval_mixed<float>;
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<(unsigned)blocks, warps * 32, smem, (cudaStream_t)stream>>>(*p);
  }
  CUDA_TRY(cudaGetLastError());
  g_launches.fetch_add(1);
  return THRL_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------ host-buffer call
// thrl_qtable_scan_host: the run range goes through in chunks; chunk c+1's upload and chunk c-1's download run on their own
// streams while chunk c is in the kernel.  Three chunk slots of device memory, the three streams and their events live in
// a per-device arena that is kept between calls (grown when a call needs more), so steady-state calls allocate nothing.
namespace {

struct HostArena {
  void* base = nullptr;
  size_t bytes = 0;
  cudaStream_t up = nullptr, run = nullptr, down = nullptr;
  cudaEvent_t ev_up[3] = {}, ev_run[3] = {}, ev_down[3] = {};
  bool ready = false;
  std::mutex mu;  // one host call per device at a time
};
HostArena g_arena[64];

// resident runs of the latest launch per game (memcmp of the laid-out ThrlGame + dtype): lets the next host call size its
// chunks in whole rounds of the persistent grid from the first chunk on
struct WaveEntry { ThrlGame g; int dtype; long long wave; };
std::vector<WaveEntry> g_waves;
std::mutex g_waves_mu;
long long wave_lookup(const ThrlGame& G, int dtype) {
  std::lock_guard<std::mutex> lock(g_waves_mu);
  for (auto& e : g_waves) if (e.dtype == dtype && memcmp(&e.g, &G, sizeof(G)) == 0) return e.wave;
  return 0;
}
void wave_store(const ThrlGame& G, int dtype, long long wave) {
  std::lock_guard<std::mutex> lock(g_waves_mu);
  for (auto& e : g_waves) if (e.dtype == dtype && memcmp(&e.g, &G, sizeof(G)) == 0) { e.wave = wave; return; }
  if (g_waves.size() >= 32) g_waves.erase(g_waves.begin());
  g_waves.push_back(WaveEntry{G, dtype, wave});
}

int arena_prepare(HostArena& A, size_t need) {
  if (!A.ready) {
    CUDA_TRY(cudaStreamCreateWithFlags(&A.up, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&A.run, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&A.down, cudaStreamNonBlocking));
    for (int k = 0; k < 3; ++k) {
      CUDA_TRY(cudaEventCreateWithFlags(&A.ev_up[k], cudaEventDisableTiming));
      CUDA_TRY(cudaEventCreateWithFlags(&A.ev_run[k], cudaEventDisableTiming));
      CUDA_TRY(cudaEventCreateWithFlags(&A.ev_down[k], cudaEventDisableTiming));
    }
    A.ready = true;
  }
  if (need > A.bytes) {
    if (A.base) CUDA_TRY(cudaFree(A.base));
    A.base = nullptr;
    A.bytes = 0;
    const size_t want = need + need / 8;  // a little headroom: chunk sizes move by a wave between calls
    if (cudaMalloc(&A.base, want) != cudaSuccess) {
      (void)cudaGetLastError();
      CUDA_TRY(cudaMalloc(&A.base, need));
      A.bytes = need;
    } else {
      A.bytes = want;
    }
  }
  return THRL_OK;
}

// Run-range boundaries of the chunks (same rule as th_rl_b200.engine.chunk_bounds): first and last chunk carry half the
// weight (their upload / download is the only copy no kernel hides); whole multiples of `wave` once the batch spans at
// least two rounds per chunk.
std::vector<long long> chunk_bounds(long long R, int n_chunks, long long wave) {
  if (n_chunks > R) n_chunks = (int)R;
  if (n_chunks < 1) n_chunks = 1;
  std::vector<int> w((size_t)n_chunks, 2);
  if (n_chunks >= 3) w.front() = w.back() = 1;
  long long tot = 0;
  for (int x : w) tot += x;
  const long long unit = (wave > 0 && (R + wave - 1) / wave >= 2LL * n_chunks) ? wave : 1;
  const long long units = (R + unit - 1) / unit;
  std::vector<long long> b{0};
  long long acc = 0;
  for (int x : w) {
    acc += x;
    long long v = units * acc / tot * unit;
    if (v > R) v = R;
    if (v < b.back()) v = b.back();
    b.push_back(v);
  }
  b.back() = R;
  return b;
}

}  // namespace

extern "C" int thrl_qtable_scan_host(const ThrlScanArgs* a, int device) {
  int rc = check_args(a);
  if (rc) return rc;
  ThrlGame G = *a->game;
  rc = validate_layout(&G);
  if (rc) return rc;
  if (G.run_stride > 0 && !a->q) return fail(THRL_ERR_BAD_ARGS, "q must not be NULL (the game has Q-tables)");
  rc = check_args_game(a, G);
  if (rc) return rc;
  if (device < 0 || device >= 64) return fail(THRL_ERR_BAD_ARGS, "device index %d", device);
  if (cudaSetDevice(device) != cudaSuccess) return fail(THRL_ERR_NO_DEVICE, "cudaSetDevice(%d) failed (there is no CPU fallback)", device);
  const long long R = a->n_runs;
  const size_t n = (size_t)G.n_agents, T = (size_t)G.max_steps, E = (size_t)(a->epoch_end - a->epoch_begin);
  if (R == 0 || E == 0) return THRL_OK;
  const size_t esz = a->table_dtype == THRL_F64 ? 8 : 4;

  // per-run bytes of every buffer that travels with a chunk: {host pointer, bytes per run, upload, download}
  struct Buf { const void* h; size_t per_run; bool in, out; size_t off; };
  enum { Q, CNT, EPS, PRICE, HP, RING, MLP, RU, RRA, RNA, TA, TR, TP, NBUF };
  Buf buf[NBUF] = {
      {a->q, (size_t)G.run_stride * esz, true, true, 0},
      {a->counter, (size_t)G.run_stride * 4, true, true, 0},
      {a->eps, n * 8, true, true, 0},
      {a->price, 8, true, true, 0},
      {a->hp, n * 32, true, false, 0},
      {G.regular ? nullptr : a->ring, (size_t)ring_bytes(&G), true, true, 0},
      {a->mlp, (size_t)G.mlp_stride * 4, true, true, 0},
      {a->replay_u, E * T * n * 8, true, false, 0},
      {a->replay_ra, E * T * n * 4, true, false, 0},
      {a->replay_new_a, E * T * 8, true, false, 0},
      {a->trace_actions, E * T * n * 4, false, true, 0},
      {a->trace_rewards, E * T * n * 8, false, true, 0},
      {a->trace_prices, E * T * 8, false, true, 0},
  };
  size_t per_run = 0;
  for (auto& b : buf) if (b.h) per_run += b.per_run;
  const size_t log_per_run = E * n * 8;  // rewards_log / actions_log: only the first n_log_runs runs of the call have a row
  const size_t statb = a->stats ? E * n * THRL_STATS_K * 8 : 0;

  // chunking: small batches go through in one piece; otherwise 12 chunks (THRL_HOST_CHUNKS overrides)
  int n_chunks = ((size_t)R * per_run < (size_t)(16u << 20)) ? 1 : 12;
  if (const char* e = getenv("THRL_HOST_CHUNKS")) if (atoi(e) >= 1) n_chunks = atoi(e);
  const std::vector<long long> bounds = chunk_bounds(R, n_chunks, wave_lookup(G, a->table_dtype));
  n_chunks = (int)bounds.size() - 1;
  long long cap = 0;
  for (int c = 0; c < n_chunks; ++c) cap = std::max(cap, bounds[c + 1] - bounds[c]);

  // slot layout for `cap` runs
  size_t slot_bytes = 0;
  for (auto& b : buf) {
    if (!b.h) continue;
    b.off = slot_bytes;
    slot_bytes += ((size_t)cap * b.per_run + 255) / 256 * 256;
  }
  size_t off_rl = 0, off_al = 0;
  if (a->rewards_log) { off_rl = slot_bytes; slot_bytes += ((size_t)std::min<long long>(cap, a->n_log_runs) * log_per_run + 255) / 256 * 256; }
  if (a->actions_log) { off_al = slot_bytes; slot_bytes += ((size_t)std::min<long long>(cap, a->n_log_runs) * log_per_run + 255) / 256 * 256; }
  const int n_slots = n_chunks < 3 ? n_chunks : 3;
  const size_t stats_off = (size_t)n_slots * slot_bytes;

  HostArena& A = g_arena[device];
  std::lock_guard<std::mutex> lock(A.mu);
  rc = arena_prepare(A, stats_off + statb + 256);
  if (rc) return rc;
  unsigned char* base = (unsigned char*)A.base;
  long long* d_stats = a->stats ? (long long*)(base + stats_off) : nullptr;
#define TRYQ(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { cudaDeviceSynchronize(); return fail(THRL_ERR_CUDA, "%s: %s", #x, cudaGetErrorString(e_)); } } while (0)
  if (a->stats) TRYQ(cudaMemcpyAsync(d_stats, a->stats, statb, cudaMemcpyHostToDevice, A.run));  // accumulated (+=) by every chunk
  long long wave = 0;
  for (int c = 0; c < n_chunks; ++c) {
    const long long b0 = bounds[c], b1 = bounds[c + 1], Rc = b1 - b0;
    if (Rc <= 0) continue;
    const int sl = c % 3;
    unsigned char* S = base + (size_t)sl * slot_bytes;
    if (c >= 3) TRYQ(cudaStreamWaitEvent(A.up, A.ev_down[sl], 0));  // the slot's previous chunk has left the device
    for (auto& b : buf)
      if (b.h && b.in)
        TRYQ(cudaMemcpyAsync(S + b.off, (const unsigned char*)b.h + (size_t)b0 * b.per_run, (size_t)Rc * b.per_run, cudaMemcpyHostToDevice, A.up));
    TRYQ(cudaEventRecord(A.ev_up[sl], A.up));
    TRYQ(cudaStreamWaitEvent(A.run, A.ev_up[sl], 0));
    if (c >= 3) TRYQ(cudaStreamWaitEvent(A.run, A.ev_down[sl], 0));  // outputs that are only written (traces, logs) share the slot too
    ThrlScanArgs d = *a;
    d.game = &G;
    d.n_runs = Rc;
    d.run_id0 = a->run_id0 + b0;
    auto dp = [&](int k) -> void* { return buf[k].h ? (void*)(S + buf[k].off) : nullptr; };
    d.q = dp(Q); d.counter = (uint32_t*)dp(CNT); d.eps = (double*)dp(EPS); d.price = (double*)dp(PRICE);
    d.hp = (const double*)dp(HP); d.ring = dp(RING); d.mlp = (float*)dp(MLP);
    d.replay_u = (const double*)dp(RU); d.replay_ra = (const int32_t*)dp(RRA); d.replay_new_a = (const double*)dp(RNA);
    d.trace_actions = (int32_t*)dp(TA); d.trace_rewards = (double*)dp(TR); d.trace_prices = (double*)dp(TP);
    const long long nlog = std::max<long long>(0, std::min<long long>(a->n_log_runs - b0, Rc));
    d.n_log_runs = nlog;
    d.rewards_log = (a->rewards_log && nlog) ? (double*)(S + off_rl) : nullptr;
    d.actions_log = (a->actions_log && nlog) ? (double*)(S + off_al) : nullptr;
    d.stats = (int64_t*)d_stats;
    rc = thrl_qtable_scan(&d, A.run);
    if (rc) { cudaDeviceSynchronize(); return rc; }
    if (g_last_wave > wave) wave = g_last_wave;
    TRYQ(cudaEventRecord(A.ev_run[sl], A.run));
    TRYQ(cudaStreamWaitEvent(A.down, A.ev_run[sl], 0));
    for (auto& b : buf)
      if (b.h && b.out)
        TRYQ(cudaMemcpyAsync((unsigned char*)b.h + (size_t)b0 * b.per_run, S + b.off, (size_t)Rc * b.per_run, cudaMemcpyDeviceToHost, A.down));
    if (d.rewards_log) TRYQ(cudaMemcpyAsync((unsigned char*)a->rewards_log + (size_t)b0 * log_per_run, S + off_rl, (size_t)nlog * log_per_run, cudaMemcpyDeviceToHost, A.down));
    if (d.actions_log) TRYQ(cudaMemcpyAsync((unsigned char*)a->actions_log + (size_t)b0 * log_per_run, S + off_al, (size_t)nlog * log_per_run, cudaMemcpyDeviceToHost, A.down));
    TRYQ(cudaEventRecord(A.ev_down[sl], A.down));
  }
  if (a->stats) TRYQ(cudaMemcpyAsync(a->stats, d_stats, statb, cudaMemcpyDeviceToHost, A.run));
  cudaError_t e1 = cudaStreamSynchronize(A.run), e2 = cudaStreamSynchronize(A.down), e3 = cudaStreamSynchronize(A.up);
#undef TRYQ
  if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess)
    return fail(THRL_ERR_CUDA, "scan failed: %s", cudaGetErrorString(e1 != cudaSuccess ? e1 : (e2 != cudaSuccess ? e2 : e3)));
  if (wave > 0) wave_store(G, a->table_dtype, wave);
  g_last_wave = wave;
  return THRL_OK;
}

extern "C" int thrl_release_device_memory(void) {
  int device = 0;
  if (cudaGetDevice(&device) != cudaSuccess || device < 0 || device >= 64) return fail(THRL_ERR_NO_DEVICE, "no CUDA device");
  HostArena& A = g_arena[device];
  {
    std::lock_guard<std::mutex> lock(A.mu);
    if (A.base) {
      CUDA_TRY(cudaDeviceSynchronize());
      CUDA_TRY(cudaFree(A.base));
      A.base = nullptr;
      A.bytes = 0;
    }
  }
  if (cudaMemPool_t pool = pwl_pool(device, false)) {
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemPoolTrimTo(pool, 0));
  }
  return THRL_OK;
}

extern "C" int thrl_curve_hist(const double* rewards_log, int64_t n_runs, int32_t epochs, int32_t n_agents, double decay,
                               const double* den, double* ewm_num, double lo, double hi, int32_t n_bins, int64_t* hist,
                               void* stream) {
  if (!rewards_log || !den || !ewm_num || !hist) return fail(THRL_ERR_BAD_ARGS, "thrl_curve_hist: NULL argument");
  if (n_runs < 0 || epochs < 0 || n_agents < 1 || n_agents > THRL_MAX_AGENTS || n_bins < 1 || !(hi > lo) || !(decay > 0.0 && decay < 1.0))
    return fail(THRL_ERR_BAD_ARGS, "thrl_curve_hist: n_runs=%lld epochs=%d n_agents=%d n_bins=%d lo=%g hi=%g decay=%g",
                (long long)n_runs, epochs, n_agents, n_bins, lo, hi, decay);
  if (n_runs == 0 || epochs == 0) return THRL_OK;
  DeviceInfo dev;
  int rc = device_info(&dev);
  if (rc) return rc;
  thrl::CurveHistParams p;
  p.rewards_log = rewards_log; p.n_runs = n_runs; p.E = epochs; p.n = n_agents;
  p.decay = decay;
  p.den = den; p.ewm_num = ewm_num; p.lo = lo; p.inv_width = (double)n_bins / (hi - lo); p.n_bins = n_bins;
  p.hist = (unsigned long long*)hist;
  const long long blocks = (n_runs + 255) / 256;
  thrl::curve_hist<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(p);
  CUDA_TRY(cudaGetLastError());
  g_launches.fetch_add(1);
  return THRL_OK;
}
