// Persistent Metropolis-Hastings loop for small data sets (BASELINE configs 1 / 2: bnn_classify.py, bnn_regress.py --
// a few thousand rows, a few hundred weights): ONE launch runs n_steps iterations of MCMC.mh_step (BNN_env.py:381-532).
//
// With two launches per iteration (k_mh_update, k_fwd_generic) a step of such a chain costs ~30 us even when replayed
// from a CUDA graph: two kernel boundaries, the proposal travelling through L2 / HBM, and a 2.5 MB feature matrix
// re-read through L2 by 40 CTAs -- for 3.5 MFLOP of arithmetic.  Here a thread-block CLUSTER owns a chain:
//   * the leader CTA (cluster rank 0) runs the update body (bnn_mh_body.cuh: accept step s-1, adapt, propose step s,
//     prior, pack) -- the same code, thread count and reduction order as k_mh_update, so chains are bit-identical;
//   * barrier.cluster (release / acquire);
//   * every CTA of the cluster copies the packed proposal into shared memory and runs the generic forward body
//     (bnn_generic_body.cuh) over its share of the 16-row tiles, whose X rows stay RESIDENT in shared memory for the
//     whole launch when they fit (config 1: 2.5 MB over 16 CTAs); per-tile partials and the accuracy counters go
//     straight into the leader's shared memory (distributed shared memory stores / atomics);
//   * barrier.cluster; next step.
// Chains are independent, so the C clusters of a launch need not be co-resident.
#include <cooperative_groups.h>
#include "bnn_mh_body.cuh"
#include "bnn_generic_body.cuh"

namespace cg = cooperative_groups;

constexpr int CL_MAX_WARPS = 16;            // warps per CTA: 8 (the update team) .. 16, as many as the tiles need

// Tile assignment.  The leader CTA also carries the chain state (weights, owner scratch, draw cache) and does the update
// while the others wait, so it takes what the worker CTAs (ranks 1 .. cluster-1) leave over:
//   worker rank r, warp w, slot i < tw :  tile (i * (cluster - 1) + r - 1) * warps + w      (if < n_worker_tiles)
//   leader, warp w, slot i < tl        :  tile n_worker_tiles + i * warps + w                (if < n_tiles16)
struct ChainLoopPlan {
  int cluster;            // CTAs per chain
  int warps;              // warps per CTA
  int tw, tl;             // tile slots per warp: workers / leader
  int n_worker_tiles;     // tiles owned by the worker CTAs
  int x_resident;         // X tiles (+ their labels / targets) kept in shared memory for the whole launch
  size_t smem;            // dynamic shared memory per CTA
};

// shared-memory carve-up in doubles.  Common prefix, the same in every CTA of the cluster (part and cnt_leader of rank 0
// are written by the other ranks through distributed shared memory):
//   tab [GEN_TAB_SIZE] | part [NF * n_tiles16] | w [PB] | alpha | stage [warps * per_warp] | cnt_leader, cnt_local (ints)
// leader only:  wstate [2P] | ddz [2][UPD_DRAW_CAP] | owner [P] (ints) | didx [2][UPD_DRAW_CAP] (ints) | pk [P] (ints)
// then the resident tiles of the CTA: per tile  X [16 * F_pad] | targets [16 * K] (Gaussian) or labels [16] (ints)
__host__ __device__ inline size_t chain_loop_per_warp(const NetGeom& g) {
  const int ZS = g.l[g.L - 1].out_pad + 1;
  return 2 * 16 * (size_t)g.max_w + 16 * (size_t)ZS;
}
__host__ __device__ inline size_t chain_loop_common_doubles(const NetGeom& g, int NF, long long nt, int warps) {
  const int NC = bnn_n_counts(g.K);
  return GEN_TAB_SIZE + (((size_t)NF * nt + 1) & ~(size_t)1) + (size_t)g.PB + ((BNN_MAX_LAYERS + 1) & ~1) +
         (size_t)warps * chain_loop_per_warp(g) + (size_t)((NC + 3) & ~3);      // (2 * NC4 ints = NC4 doubles)
}
__host__ __device__ inline size_t chain_loop_leader_doubles(const NetGeom& g) {
  return 2 * (size_t)((g.P + 1) & ~1) + 2 * UPD_DRAW_CAP + (size_t)((g.P + 3) & ~3) + UPD_DRAW_CAP;
}
__host__ __device__ inline size_t chain_loop_tile_doubles(const NetGeom& g) {
  return 16 * (size_t)g.F_pad + (g.lik == BNN_LIK_CATEGORICAL ? 8 : 16 * (size_t)g.K);
}

template <int ACT, bool XRES>
__global__ void __launch_bounds__(CL_MAX_WARPS * 32, 1) k_chain_loop(const __grid_constant__ ChainDev d,
                                                                      const __grid_constant__ FwdParams p0, int n_steps,
                                                                      int tw, int tl, int n_worker_tiles) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ FwdParams sp;                  // this chain's forward parameters (partials -> the leader's shared memory)
  cg::cluster_group cluster = cg::this_cluster();
  const int CL = (int)cluster.dim_blocks().x;
  const int rank = (int)cluster.block_rank();
  const int c = (int)(blockIdx.x / CL);
  const NetGeom& g = d.g;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int NTHR = (int)blockDim.x, NW = NTHR >> 5;
  const int gq = lane >> 2;
  const int NC = bnn_n_counts(g.K), NC4 = (NC + 3) & ~3;
  const int ZS = g.l[g.L - 1].out_pad + 1;
  const long long nt = d.n_tiles16;
  const bool leader = (rank == 0);
  const bool cat = (g.lik == BNN_LIK_CATEGORICAL);

  double* tab = reinterpret_cast<double*>(smem_raw);
  double* part_sm = tab + GEN_TAB_SIZE;
  double* wsm = part_sm + (((size_t)d.NF * nt + 1) & ~(size_t)1);
  double* alpha_sm = wsm + g.PB;
  double* stage = alpha_sm + ((BNN_MAX_LAYERS + 1) & ~1);                // 16-byte aligned: double2 accesses
  const size_t per_warp = chain_loop_per_warp(g);
  double* h0 = stage + warp * per_warp;
  double* h1 = h0 + 16 * g.max_w;
  double* zs = h1 + 16 * g.max_w;
  int* cnt_leader = reinterpret_cast<int*>(stage + NW * per_warp);
  int* cnt_local = cnt_leader + NC4;
  double* role = reinterpret_cast<double*>(cnt_local + NC4);
  // leader only
  double* wstate = role;                                                 // [2P] current | proposed weights
  double* ddz_sm = wstate + 2 * (size_t)((g.P + 1) & ~1);
  int* owner_sm = reinterpret_cast<int*>(ddz_sm + 2 * UPD_DRAW_CAP);
  int* didx_sm = owner_sm + ((g.P + 3) & ~3);
  int* pk_sm = didx_sm + 2 * UPD_DRAW_CAP;
  double* xsm = leader ? role + chain_loop_leader_doubles(g) : role;
  const size_t tile_d = chain_loop_tile_doubles(g);

  double* part_leader = cluster.map_shared_rank(part_sm, 0);
  int* cnt_dst = cluster.map_shared_rank(cnt_leader, 0);

  for (int i = tid; i < GEN_TAB_SIZE; i += NTHR) tab[i] = p0.exp_tab_small[i];
  for (int i = tid; i < g.PB; i += NTHR) wsm[i] = 0.0;      // padding entries of the packed set stay zero
  if (tid == 0) {
    sp = p0;
    sp.C = 1;
    sp.part = part_leader;
    sp.counts = nullptr;
    sp.wp = wsm;
    sp.alpha = alpha_sm;
  }
  const int n_slots = leader ? tl : tw;
  auto tile_of = [&](int i) -> long long {
    if (leader) return (long long)n_worker_tiles + (long long)i * NW + warp;
    const long long t = ((long long)i * (CL - 1) + (rank - 1)) * NW + warp;
    return t < n_worker_tiles ? t : nt;
  };
  if (XRES) {
    // the rows of the tiles this warp owns, once per launch (global layout == shared layout: swizzled rows)
    for (int i = 0; i < n_slots; ++i) {
      const long long wt = tile_of(i);
      if (wt >= nt) break;
      double* slot = xsm + ((size_t)i * NW + warp) * tile_d;
      const double2* src = reinterpret_cast<const double2*>(p0.x + wt * 16 * (long long)g.F_pad);
      double2* dst = reinterpret_cast<double2*>(slot);
      for (int e = lane; e < 8 * g.F_pad; e += 32) dst[e] = __ldg(src + e);
      if (cat) {
        int* lab = reinterpret_cast<int*>(slot + 16 * g.F_pad);
        if (lane < 16) lab[lane] = (wt * 16 + lane < p0.n_total) ? p0.labels[wt * 16 + lane] : 0;
      } else {
        double* tg = slot + 16 * g.F_pad;
        for (int e = lane; e < 16 * g.K; e += 32)
          tg[e] = (wt * 16 + e / g.K < p0.n_total) ? p0.targets[wt * 16 * g.K + e] : 0.0;
      }
    }
  }
  __syncthreads();
  const FwdParams& p = sp;
  UpdLoop ctx;
  ctx.part_c = part_sm; ctx.counts_c = cnt_leader; ctx.w_sm = wstate; ctx.owner_sm = owner_sm; ctx.wpk_sm = wsm;
  ctx.didx_sm = didx_sm; ctx.ddz_sm = ddz_sm; ctx.pk_sm = pk_sm;
  const double2* wsrc = reinterpret_cast<const double2*>(d.wp_prop + (long long)c * g.PB);

  for (int s = 0; s <= n_steps; ++s) {
    // leader CTA, first UPD_TEAM_THREADS threads: accept step s-1, propose step s (the packed proposal lands in wsm)
    if (leader && tid < UPD_TEAM_THREADS) {
      ctx.first = (s == 0); ctx.last = (s == n_steps);
      mh_update_body<true>(d, c, s > 0 ? 1 : 0, s < n_steps ? 1 : 0, s, ctx);
      if (s < n_steps && tid < g.L) alpha_sm[tid] = d.alpha_fwd[(long long)c * g.L + tid];   // written by thread 0 before the team's last barrier
    }
    if (s == n_steps) break;
    cluster.sync();                          // the proposal of step s (packed weights, slopes, zeroed counters) is visible
    if (!leader) {
      // packed proposal from L2 (a pull from the leader's shared memory by 15 CTAs at once is bound by that SM's
      // shared-memory port: 5.7k clk measured against 2k through L2)
      for (int i = tid; i < g.PB / 2; i += NTHR) reinterpret_cast<double2*>(wsm)[i] = __ldcg(wsrc + i);
      if (tid < g.L) alpha_sm[tid] = __ldcg(d.alpha_fwd + (long long)c * g.L + tid);
    }
    for (int i = tid; i < NC; i += NTHR) cnt_local[i] = 0;
    __syncthreads();
    for (int i = 0; i < n_slots; ++i) {
      const long long wt = tile_of(i);
      if (wt >= nt) break;
      const double* slot = xsm + ((size_t)i * NW + warp) * tile_d;
      const double* xt = XRES ? slot : p.x + wt * 16 * (long long)g.F_pad;
      const double* xrow0 = xt + gq * g.F_pad;
      const double* xrow1 = xrow0 + 8 * g.F_pad;
      fwd_generic_layers<ACT, !XRES, false>(g, xrow0, xrow1, wsm, (ACT == BNN_ACT_LEAKY) ? alpha_sm : nullptr, h0, h1, zs,
                                            ZS, tab, lane);
      bnn_epilogue<false, false, GEN_TB>(p, 0, wt, lane, zs, ZS, tab, cnt_local, nullptr, nullptr,
                                         (XRES && cat) ? reinterpret_cast<const int*>(slot + 16 * g.F_pad) : nullptr,
                                         (XRES && !cat) ? slot + 16 * g.F_pad : nullptr);
      __syncwarp();
    }
    // the leader's team is done with its few tiles long before the workers: it pre-proposes iteration s + 1 (layer
    // choice, scalar draws, the proposal's draws) in the time it would otherwise wait at the barrier
    if (leader && tid < UPD_TEAM_THREADS && s + 1 < n_steps) {
      ctx.first = false; ctx.last = false;
      mh_update_body<true>(d, c, 0, 3, s + 1, ctx);
    }
    __syncthreads();
    if (cat)
      for (int i = tid; i < NC; i += NTHR)
        if (cnt_local[i]) atomicAdd(&cnt_dst[i], cnt_local[i]);
    cluster.sync();                          // partials and counters of step s are in the leader's shared memory
  }
  // no CTA may exit while others can still address its shared memory
  cluster.sync();
}

// static shared memory of the kernel (update-body staging, FwdParams): the same for every instantiation up to a few bytes
static size_t chain_loop_static_smem() {
  static size_t v = 0;
  if (!v) {
    cudaFuncAttributes a{};
    if (cudaFuncGetAttributes(&a, k_chain_loop<BNN_ACT_TANH, true>) != cudaSuccess) { cudaGetLastError(); return 16384; }
    v = a.sharedSizeBytes + 256;
  }
  return v;
}

// dynamic shared memory a CTA of the kernel may use: what the static part leaves of BNN_MAX_DYN_SMEM
static size_t chain_loop_max_dyn_smem() { return BNN_MAX_DYN_SMEM - chain_loop_static_smem(); }
template <typename Kern>
static cudaError_t prepare_chain_loop(Kern kern) {
  return bnn_prepare_kernel((const void*)kern, (int)chain_loop_max_dyn_smem(), true);
}

// clusters of `cl` CTAs (warps * 32 threads, smem bytes each) the GPU can hold at the same time; cached per shape
static int chain_loop_max_clusters(int cl, int warps, size_t smem) {
  struct Key { int cl, warps; size_t smem; int n; };
  static Key cache[16];
  static int n_cache = 0;
  for (int i = 0; i < n_cache; ++i)
    if (cache[i].cl == cl && cache[i].warps == warps && cache[i].smem == smem) return cache[i].n;
  auto kern = k_chain_loop<BNN_ACT_TANH, true>;          // (every instantiation has the same footprint up to a few registers)
  if (prepare_chain_loop(kern) != cudaSuccess) { cudaGetLastError(); return 0; }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)cl);
  cfg.blockDim = dim3((unsigned)warps * 32);
  cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = (unsigned)cl; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) { cudaGetLastError(); n = 0; }
  if (n_cache < 16) cache[n_cache++] = Key{cl, warps, smem, n};
  return n;
}

// The tile assignment of one cluster size: warps per CTA, tile slots, residency.
static bool chain_loop_plan_for(const NetGeom& g, int NF, long long nt, int cl, ChainLoopPlan* plan) {
  const size_t cap = chain_loop_max_dyn_smem() / sizeof(double);
  const size_t tile_d = chain_loop_tile_doubles(g), lead_d = chain_loop_leader_doubles(g);
  const int workers = cl - 1;
  ChainLoopPlan best{};
  bool have = false;
  for (int warps = 8; warps <= CL_MAX_WARPS; ++warps) {
    const size_t common = chain_loop_common_doubles(g, NF, nt, warps);
    if (common + lead_d > cap) break;
    // tile slots per warp that fit next to the rest: workers / leader
    const long long tw_max = workers ? (long long)((cap - common) / tile_d) / warps : 0;
    const long long tl_cap = (long long)((cap - common - lead_d) / tile_d);          // leader: tiles, not slots
    for (int t = 1; t <= 8; ++t) {
      // workers take t tiles per warp, the leader at most as many (it also runs the update)
      const long long wtiles = workers ? ((long long)workers * warps * t < nt ? (long long)workers * warps * t : nt) : 0;
      const long long left = nt - wtiles;
      if (left > (long long)warps * t) continue;
      ChainLoopPlan q{};
      q.cluster = cl; q.warps = warps; q.tw = workers ? t : 0; q.tl = (int)((left + warps - 1) / warps);
      q.n_worker_tiles = (int)wtiles;
      q.x_resident = (!workers || t <= tw_max) && left <= tl_cap;
      const size_t wneed = common + (q.x_resident && workers ? (size_t)warps * t * tile_d : 0);
      const size_t lneed = common + lead_d + (q.x_resident ? (size_t)left * tile_d : 0);
      q.smem = (wneed > lneed ? wneed : lneed) * sizeof(double);
      // prefer: resident, then fewer tiles per warp (the critical path), then fewer warps
      const bool better = !have || (q.x_resident > best.x_resident) ||
                          (q.x_resident == best.x_resident && (q.tw > 0 ? q.tw : q.tl) < (best.tw > 0 ? best.tw : best.tl));
      if (better) { best = q; have = true; }
      break;                                  // the smallest t that covers the tiles at this warp count
    }
  }
  if (have) *plan = best;
  return have;
}

// mode 1 (automatic): the persistent loop is taken only where it beats the per-step launch sequence.  Measured on a B200
// (tools/loop_threshold.py, profiles/r02_chain_loop_threshold.json: [5,5] tanh network, 128 features, 500 - 30,000 rows x
// 1 - 32 chains, us per MH step):
//   loop      8 + 4.7 * tiles per warp with X resident in shared memory, 12 + 8 * tiles per warp with X streamed from L2,
//             times the number of WAVES of clusters -- so every chain's cluster must be resident at once;
//   sequence  21.5 + 0.006 * max(0, (16-row tiles) * chains - 1500).
// The largest cluster size whose C clusters fit the GPU together is planned; mode 2 (tests) skips both conditions.
static bool chain_loop_plan(const NetGeom& g, int NF, long long nt, int C, int n_sms, int max_cluster, int mode,
                            ChainLoopPlan* plan) {
  if (g.P > 2048 || nt < 1 || nt >= 4096 || g.PB % 2) return false;      // (k_mh_update would run 1,024 threads / slice partials)
  // CTAs per chain: no more than there are tiles for (one tile per warp at 8 warps), within the GPU when all chains run at once
  int cl = 16;
  while (cl > 1 && (cl > max_cluster || (long long)(cl / 2) * 8 >= nt || (long long)C * cl > n_sms)) cl >>= 1;
  for (; cl >= 1; cl >>= 1) {
    ChainLoopPlan q;
    if (!chain_loop_plan_for(g, NF, nt, cl, &q)) { if (mode >= 2) return false; continue; }
    if (mode >= 2) { *plan = q; return true; }
    if (chain_loop_max_clusters(q.cluster, q.warps, q.smem) < C) continue;           // more than one wave: try smaller clusters
    const int tpw = q.tw > q.tl ? q.tw : q.tl;
    const double loop_us = q.x_resident ? 8.0 + 4.7 * tpw : 12.0 + 8.0 * tpw;
    const double tc = (double)nt * C;
    const double seq_us = 21.5 + 0.006 * (tc > 1500.0 ? tc - 1500.0 : 0.0);
    if (loop_us < 0.95 * seq_us) { *plan = q; return true; }
    return false;
  }
  return false;
}

bool bnn_chain_loop_fits(const NetGeom& g, int NF, long long nt, int C, int n_sms, int max_cluster, int mode) {
  ChainLoopPlan plan;
  return chain_loop_plan(g, NF, nt, C, n_sms, max_cluster, mode, &plan);
}

template <int ACT, bool XRES>
static cudaError_t launch_chain_loop_t(const ChainDev& d, const FwdParams& p, int n_steps, const ChainLoopPlan& plan,
                                       cudaStream_t st) {
  auto kern = k_chain_loop<ACT, XRES>;
  if (cudaError_t e = prepare_chain_loop(kern)) return e;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(d.C * plan.cluster));
  cfg.blockDim = dim3((unsigned)plan.warps * 32);
  cfg.dynamicSmemBytes = plan.smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = (unsigned)plan.cluster;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  int tw = plan.tw, tl = plan.tl, nwt = plan.n_worker_tiles;
  return cudaLaunchKernelEx(&cfg, kern, d, p, n_steps, tw, tl, nwt);
}

template <int ACT>
static cudaError_t launch_chain_loop_a(const ChainDev& d, const FwdParams& p, int n_steps, const ChainLoopPlan& plan,
                                       cudaStream_t st) {
  return plan.x_resident ? launch_chain_loop_t<ACT, true>(d, p, n_steps, plan, st)
                         : launch_chain_loop_t<ACT, false>(d, p, n_steps, plan, st);
}

// n_steps MH iterations of every chain of d in one launch; cudaErrorNotSupported when the problem does not fit the
// persistent path (the caller then issues the per-step launch sequence)
cudaError_t bnn_launch_chain_loop(const ChainDev& d, const FwdParams& p, int n_steps, int n_sms, int max_cluster, int mode,
                                  cudaStream_t st, int* cluster_out) {
  ChainLoopPlan plan;
  if (!chain_loop_plan(d.g, d.NF, d.n_tiles16, d.C, n_sms, max_cluster, mode, &plan)) return cudaErrorNotSupported;
  if (cluster_out) *cluster_out = plan.cluster;
  return bnn_with_act(d.g.act, [&](auto a) { return launch_chain_loop_a<decltype(a)::value>(d, p, n_steps, plan, st); });
}
