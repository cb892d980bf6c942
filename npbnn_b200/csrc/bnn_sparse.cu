// Block-masked networks (create_mask, BNN_lib.py:16-47; apply_mask, BNN_env.py:259-267): the dataflow program that
// covers a mask with small dense blocks, its builder, the kernels that run it (k_fwd_sparse, k_fwd_pairs) and their
// launchers.
#include <vector>
#include "bnn_kernels.h"
#include "bnn_generic_body.cuh"

// A masked hidden layer is a list of small dense blocks ("items": rows r0..r0+nr-1, nr <= 4, columns
// c0..c0+nc-1) that cover every entry the mask keeps; entries outside the blocks are exactly zero in every
// proposal (w' *= mask, BNN_env.py:461-462), so skipping them changes nothing but the order of the sum.
// At the block sizes create_mask produces (a feature feeds a handful of nodes) the contraction is far too
// thin for tensor-core tiles and the FP64 work is dominated by the activations, so this kernel is plain DFMA
// with one THREAD per row: lane = row of a 32-row tile, every lane runs the same item, weights are warp-
// uniform shared-memory loads.  The host (bnn_sparse_build, below) orders the items of all hidden
// layers as a dataflow program -- an item runs as soon as the units it reads exist -- and assigns each hidden
// unit a scratch slot that is recycled after its last reader, so a thread needs F + (live units) doubles of
// shared memory instead of every layer's width; the units of the LAST hidden layer are never stored: they are
// multiplied into the (dense, O <= 8) output layer's accumulators, which stay in registers.
//   * the weights the program touches are gathered once per CTA from the packed weight sets into shared
//     memory IN PROGRAM ORDER (sp.widx), so the item loop reads them with a running pointer and 16-byte
//     loads -- no address arithmetic per multiply-add;
//   * four (or two) chains are evaluated together (same program, different weights) for instruction-level
//     parallelism;
//   * a work unit is (32-row tile, chain subset); a CTA owns a contiguous range of tiles and its warps draw
//     units from a shared counter, so the load is balanced to one unit.
//
// program (ints), per item: [0] layer | nr << 8 | to_out << 16  [1] nc  [2] 1 if the inputs are scratch slots
//     (0: X columns, shared by both chains)  [3] 0  [4..7] element offset of each produced unit's slot
//     [8..8+nc) element offset of each input, padded to a multiple of 4 ints (offsets are for the first chain of the unit; chain q's
//     scratch slots follow q * sp.slots * SP_US elements later)
// weight stream (doubles), per chain: [0..8) output-layer bias; then per item: bias[nrp], nc x w[nrp] (column
//     c0+k, rows r0..r0+nr-1) and, for to_out items, nr x w_out[op] (the output-layer column of each produced
//     unit); nrp / op = nr / O rounded up to even, padding is 0.
constexpr int SP_US = 33;        // per-unit stride in doubles (32 rows + 1: conflict-free transposed stores)
constexpr int SP_MAX_O = 8;
constexpr int SP_HDR = 8;

template <int ACT, int NCH, int NR>
__device__ __forceinline__ void sparse_item(const int* it, int nc, int qs, int sq, bool to_out, int O,
                                            const double* (&w)[NCH], double* bufl, const double (&alpha)[NCH],
                                            const double* tab, double (&out)[NCH][SP_MAX_O]) {
  constexpr int NRP = (NR + 1) & ~1;
  double acc[NCH][NRP];
#pragma unroll
  for (int q = 0; q < NCH; ++q)
#pragma unroll
    for (int i = 0; i < NRP; i += 2) {
      const double2 b = *reinterpret_cast<const double2*>(w[q] + i);
      acc[q][i] = b.x; acc[q][i + 1] = b.y;
    }
#pragma unroll 2
  for (int k = 0; k < nc; ++k) {
    const int src = it[SP_HDR + k];
#pragma unroll
    for (int q = 0; q < NCH; ++q) {
      const double a = bufl[src + q * qs];
#pragma unroll
      for (int i = 0; i < NRP; i += 2) {
        const double2 ww = *reinterpret_cast<const double2*>(w[q] + (k + 1) * NRP + i);
        acc[q][i] = fma(ww.x, a, acc[q][i]);
        if (i + 1 < NR) acc[q][i + 1] = fma(ww.y, a, acc[q][i + 1]);
      }
    }
  }
  bool care = false;
#pragma unroll
  for (int q = 0; q < NCH; ++q)
#pragma unroll
    for (int i = 0; i < NR; ++i) care |= bnn_act_needs_care<ACT>(acc[q][i]);
  if (!__any_sync(FULL_MASK, care)) {
#pragma unroll
    for (int q = 0; q < NCH; ++q)
#pragma unroll
      for (int i = 0; i < NR; ++i) acc[q][i] = bnn_act_fast<ACT>(acc[q][i], alpha[q], tab);
  } else {
#pragma unroll
    for (int q = 0; q < NCH; ++q)
#pragma unroll
      for (int i = 0; i < NR; ++i) acc[q][i] = bnn_act<ACT>(acc[q][i], alpha[q], tab);
  }
  int adv = (nc + 1) * NRP;
  if (to_out) {
    const int op = (O + 1) & ~1;
#pragma unroll
    for (int i = 0; i < NR; ++i) {
#pragma unroll
      for (int j = 0; j < SP_MAX_O / 2; ++j) {
        if (2 * j < O) {
#pragma unroll
          for (int q = 0; q < NCH; ++q) {
            const double2 ww = *reinterpret_cast<const double2*>(w[q] + adv + i * op + 2 * j);
            out[q][2 * j] = fma(ww.x, acc[q][i], out[q][2 * j]);
            out[q][2 * j + 1] = fma(ww.y, acc[q][i], out[q][2 * j + 1]);
          }
        }
      }
    }
    adv += NR * op;
  } else {
    const int4 sl = *reinterpret_cast<const int4*>(it + 4);
    const int slot[4] = {sl.x, sl.y, sl.z, sl.w};
#pragma unroll
    for (int q = 0; q < NCH; ++q)
#pragma unroll
      for (int i = 0; i < NR; ++i) bufl[slot[i] + q * sq] = acc[q][i];
  }
#pragma unroll
  for (int q = 0; q < NCH; ++q) w[q] += adv;
}

// Fused evaluation of one "block pair" for networks whose program is a uniform sequence of pairs (what create_mask
// produces when every feature group has the same node counts, BASELINE config 3: 40 x [1 feature -> 3 nodes -> 2
// nodes]): a first-layer item (NR1 units reading nc1 features) directly followed by the second-layer item that reads
// exactly those units (NR2 units, feeding the output layer).  Same program, same weight stream as the interpreter
// (sparse_item), but the hidden units stay in registers (no scratch slots), the item headers are not decoded and
// there is no dispatch on the item height -- the interpreter spends two thirds of its instructions on those.
template <int ACT, int NCH, int NR1, int NR2, int NC1 = 0>
__device__ __forceinline__ void sparse_pair(const int* it, int nc1_rt, int O, const double* (&w)[NCH], const double* bufl,
                                            const double (&alpha1)[NCH], const double (&alpha2)[NCH], const double* tab,
                                            double (&out)[NCH][SP_MAX_O]) {
  constexpr int P1 = (NR1 + 1) & ~1, P2 = (NR2 + 1) & ~1;
  double h1[NCH][P1], h2[NCH][P2];
#pragma unroll
  for (int q = 0; q < NCH; ++q)
#pragma unroll
    for (int i = 0; i < P1; i += 2) {
      const double2 b = *reinterpret_cast<const double2*>(w[q] + i);
      h1[q][i] = b.x; h1[q][i + 1] = b.y;
    }
  const int nc1 = NC1 > 0 ? NC1 : nc1_rt;                    // NC1 > 0: features per pair known at compile time
#pragma unroll
  for (int k = 0; k < nc1; ++k) {
    const double a = bufl[it[SP_HDR + k]];                   // the feature is shared by the chains
#pragma unroll
    for (int q = 0; q < NCH; ++q)
#pragma unroll
      for (int i = 0; i < P1; i += 2) {
        const double2 ww = *reinterpret_cast<const double2*>(w[q] + (k + 1) * P1 + i);
        h1[q][i] = fma(ww.x, a, h1[q][i]);
        if (i + 1 < NR1) h1[q][i + 1] = fma(ww.y, a, h1[q][i + 1]);
      }
  }
  const int adv1 = (nc1 + 1) * P1;
  bool care = false;
#pragma unroll
  for (int q = 0; q < NCH; ++q)
#pragma unroll
    for (int i = 0; i < NR1; ++i) care |= bnn_act_needs_care<ACT>(h1[q][i]);
  if (!__any_sync(FULL_MASK, care)) {
#pragma unroll
    for (int q = 0; q < NCH; ++q)
#pragma unroll
      for (int i = 0; i < NR1; ++i) h1[q][i] = bnn_act_fast<ACT>(h1[q][i], alpha1[q], tab);
  } else {
#pragma unroll
    for (int q = 0; q < NCH; ++q)
#pragma unroll
      for (int i = 0; i < NR1; ++i) h1[q][i] = bnn_act<ACT>(h1[q][i], alpha1[q], tab);
  }
  // second-layer item: bias[P2], then one column of P2 weights per first-layer unit
#pragma unroll
  for (int q = 0; q < NCH; ++q)
#pragma unroll
    for (int j = 0; j < P2; j += 2) {
      const double2 b = *reinterpret_cast<const double2*>(w[q] + adv1 + j);
      h2[q][j] = b.x; h2[q][j + 1] = b.y;
    }
#pragma unroll
  for (int i = 0; i < NR1; ++i)
#pragma unroll
    for (int q = 0; q < NCH; ++q)
#pragma unroll
      for (int j = 0; j < P2; j += 2) {
        const double2 ww = *reinterpret_cast<const double2*>(w[q] + adv1 + (i + 1) * P2 + j);
        h2[q][j] = fma(ww.x, h1[q][i], h2[q][j]);
        if (j + 1 < NR2) h2[q][j + 1] = fma(ww.y, h1[q][i], h2[q][j + 1]);
      }
  care = false;
#pragma unroll
  for (int q = 0; q < NCH; ++q)
#pragma unroll
    for (int j = 0; j < NR2; ++j) care |= bnn_act_needs_care<ACT>(h2[q][j]);
  if (!__any_sync(FULL_MASK, care)) {
#pragma unroll
    for (int q = 0; q < NCH; ++q)
#pragma unroll
      for (int j = 0; j < NR2; ++j) h2[q][j] = bnn_act_fast<ACT>(h2[q][j], alpha2[q], tab);
  } else {
#pragma unroll
    for (int q = 0; q < NCH; ++q)
#pragma unroll
      for (int j = 0; j < NR2; ++j) h2[q][j] = bnn_act<ACT>(h2[q][j], alpha2[q], tab);
  }
  const int adv2 = adv1 + (NR1 + 1) * P2;
  const int op = (O + 1) & ~1;
#pragma unroll
  for (int j = 0; j < NR2; ++j)
#pragma unroll
    for (int o = 0; o < SP_MAX_O / 2; ++o)
      if (2 * o < O) {
#pragma unroll
        for (int q = 0; q < NCH; ++q) {
          const double2 ww = *reinterpret_cast<const double2*>(w[q] + adv2 + j * op + 2 * o);
          out[q][2 * o] = fma(ww.x, h2[q][j], out[q][2 * o]);
          out[q][2 * o + 1] = fma(ww.y, h2[q][j], out[q][2 * o + 1]);
        }
      }
#pragma unroll
  for (int q = 0; q < NCH; ++q) w[q] += adv2 + NR2 * op;
}

// NCH chains per work unit: 4 (at most 10 warps, <= 204 registers) or 2 (at most 16 warps, <= 128 registers).
template <int ACT, int NCH>
__global__ void __launch_bounds__(NCH == 4 ? 320 : 512, 1) k_fwd_sparse(const __grid_constant__ FwdParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const NetGeom& g = p.g;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  constexpr int ZS = SP_MAX_O + 1;
  const int O = g.O;
  const int G = p.sp.group;                                   // chains whose weight streams are resident
  const int sq = p.sp.slots * SP_US;

  double* tab = reinterpret_cast<double*>(smem_raw);
  double* wsm = tab + BNN_EXP_TAB_SIZE;                       // [G][sp.wlen]
  const int per_warp = (g.F + NCH * p.sp.slots) * SP_US + 32 * ZS;
  double* buf = wsm + (size_t)G * p.sp.wlen + warp * per_warp;
  double* zs = buf + (g.F + NCH * p.sp.slots) * SP_US;
  int* cnt = reinterpret_cast<int*>(wsm + (size_t)G * p.sp.wlen + nwarps * per_warp);
  const int n_cnt = bnn_smem_counts(g, p.C);
  int* next_unit = cnt + n_cnt;
  int* prog = reinterpret_cast<int*>((reinterpret_cast<uintptr_t>(next_unit + 1) + 15) & ~(uintptr_t)15);

  for (int i = threadIdx.x; i < BNN_EXP_TAB_SIZE; i += blockDim.x) tab[i] = p.exp_tab[i];
  for (int i = threadIdx.x; i < n_cnt; i += blockDim.x) cnt[i] = 0;
  for (int i = threadIdx.x; i < p.sp.prog_len; i += blockDim.x) prog[i] = p.sp.prog[i];

  // this CTA's contiguous range of 32-row tiles
  const long long n_tiles32 = (p.n_tiles16 + 1) >> 1;
  const long long n_pad = p.n_tiles16 * 16;
  const long long t0 = n_tiles32 * blockIdx.x / gridDim.x, t1 = n_tiles32 * (blockIdx.x + 1) / gridDim.x;
  double* bufl = buf + lane;

  for (int c0 = 0; c0 < p.C; c0 += G) {
    const int gc = min(G, p.C - c0);                          // chains of this group
    const int n_sub = (gc + NCH - 1) / NCH;                   // chain subsets of NCH
    __syncthreads();                                           // previous group's readers are done
    for (int i = threadIdx.x; i < gc * p.sp.wlen; i += blockDim.x) {
      const int c = i / p.sp.wlen, j = i - c * p.sp.wlen;
      const int idx = __ldg(p.sp.widx + j);
      wsm[i] = idx < 0 ? 0.0 : __ldg(p.wp + (long long)(c0 + c) * g.PB + idx);
    }
    if (threadIdx.x == 0) *next_unit = 0;
    __syncthreads();
    const int n_units = (int)(t1 - t0) * n_sub;
    long long cur_tile = -1;
    for (;;) {
      int u = 0;
      if (lane == 0) u = atomicAdd(next_unit, 1);
      u = __shfl_sync(FULL_MASK, u, 0);
      if (u >= n_units) break;
      const long long w32 = t0 + u / n_sub;
      const int sub = u - (int)(w32 - t0) * n_sub;
      if (w32 != cur_tile) {
        // X tile -> [feature][row]; global reads are contiguous (32 * F_pad consecutive doubles)
        const double* xt = p.x + w32 * 32 * (long long)g.F_pad;
        __syncwarp();
        // 8 independent loads in flight per lane (F_pad is a multiple of 8)
        for (int j0 = 0; j0 < g.F_pad; j0 += 8) {
          double v[8];
#pragma unroll
          for (int uu = 0; uu < 8; ++uu) {
            const int idx = (j0 + uu) * 32 + lane;
            v[uu] = (w32 * 32 + idx / g.F_pad < n_pad) ? __ldg(xt + idx) : 0.0;
          }
#pragma unroll
          for (int uu = 0; uu < 8; ++uu) {
            const int idx = (j0 + uu) * 32 + lane;
            const int r = idx / g.F_pad, cp = idx - r * g.F_pad;
            const int cidx = cp ^ ((r & 1) * g.x_swz);
            if (cidx < g.F) buf[cidx * SP_US + r] = v[uu];
          }
        }
        __syncwarp();
        cur_tile = w32;
      }
      // chains of this unit (a short last subset repeats its last chain; the copies are not scored)
      int ch[NCH];
      const double* w[NCH];
      double out[NCH][SP_MAX_O];
#pragma unroll
      for (int q = 0; q < NCH; ++q) {
        ch[q] = min(NCH * sub + q, gc - 1);
        w[q] = wsm + (size_t)ch[q] * p.sp.wlen;
#pragma unroll
        for (int o = 0; o < SP_MAX_O; ++o) out[q][o] = w[q][o];
        w[q] += SP_MAX_O;
      }
      const int* it = prog;
      for (int n = 0; n < p.sp.n_items; ++n) {
        const int4 h = *reinterpret_cast<const int4*>(it);
        const int layer = h.x & 0xff, nr = (h.x >> 8) & 0xff, nc = h.y;
        const bool to_out = (h.x >> 16) & 1;
        const int qs = h.z ? sq : 0;
        double alpha[NCH];
#pragma unroll
        for (int q = 0; q < NCH; ++q)
          alpha[q] = (ACT == BNN_ACT_LEAKY && p.alpha) ? p.alpha[(c0 + ch[q]) * g.L + layer] : 0.0;
        switch (nr) {
          case 1: sparse_item<ACT, NCH, 1>(it, nc, qs, sq, to_out, O, w, bufl, alpha, tab, out); break;
          case 2: sparse_item<ACT, NCH, 2>(it, nc, qs, sq, to_out, O, w, bufl, alpha, tab, out); break;
          case 3: sparse_item<ACT, NCH, 3>(it, nc, qs, sq, to_out, O, w, bufl, alpha, tab, out); break;
          default: sparse_item<ACT, NCH, 4>(it, nc, qs, sq, to_out, O, w, bufl, alpha, tab, out); break;
        }
        it += SP_HDR + ((nc + 3) & ~3);         // items are padded to 16 bytes
      }
#pragma unroll
      for (int q = 0; q < NCH; ++q) {
        if (NCH * sub + q < gc) {
          __syncwarp();
#pragma unroll
          for (int o = 0; o < SP_MAX_O; ++o) zs[lane * ZS + o] = out[q][o];
          __syncwarp();
          bnn_epilogue<false, true>(p, c0 + ch[q], w32 * 2, lane, zs, ZS, tab, cnt, nullptr, nullptr);
        }
      }
    }
  }
  if (n_cnt) {
    __syncthreads();
    for (int i = threadIdx.x; i < n_cnt; i += blockDim.x)
      if (cnt[i]) atomicAdd(&p.counts[i], cnt[i]);
  }
}

// Uniform block pairs (sparse_pair) for all chains of the pass.  Thread = row as in k_fwd_sparse, but the in-flight
// work comes from MANY warps with few chains each instead of few warps with four chains each: groups of GW warps
// share one transposed X tile (the tile's rows are the same for every chain subset), so a warp's private shared
// memory is only the 32 x 9 staging area of the likelihood epilogue and 16-24 warps fit next to the weight streams.
//   NCH 1: up to 24 warps (<= 80 registers), 2: up to 16 warps (<= 128 registers)
// Measured at BASELINE config 3 (8 chains, 200k rows): interpreter 0.90 ms per step, pairs with 4 chains x 10 warps
// 0.69, 1 chain x 24 warps 0.67, 2 chains x 16 warps 0.63 (issue slots 65 % busy, FP64 pipe 52 %).
template <int ACT, int NCH, int NR1, int NR2, int NC1>
__global__ void __launch_bounds__(NCH == 1 ? 768 : 512, 1) k_fwd_pairs(const __grid_constant__ FwdParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const NetGeom& g = p.g;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  constexpr int ZS = SP_MAX_O + 1;
  const int O = g.O;
  const int G = p.sp.group;                                   // chains whose weight streams are resident
  const int GW = p.sp.share;                                   // warps per group (share one X tile)
  const int n_groups = nwarps / GW, grp = warp / GW, wi = warp - grp * GW;

  double* tab = reinterpret_cast<double*>(smem_raw);
  double* wsm = tab + BNN_EXP_TAB_SIZE;                       // [G][sp.wlen]
  double* tile = wsm + (size_t)G * p.sp.wlen + (size_t)grp * g.F * SP_US;       // [n_groups][F][33]
  double* zs = wsm + (size_t)G * p.sp.wlen + (size_t)n_groups * g.F * SP_US + (size_t)warp * 32 * ZS;
  int* cnt = reinterpret_cast<int*>(wsm + (size_t)G * p.sp.wlen + (size_t)n_groups * g.F * SP_US + (size_t)nwarps * 32 * ZS);
  const int n_cnt = bnn_smem_counts(g, p.C);
  int* prog = cnt + ((n_cnt + 3) & ~3);                        // 16-byte aligned: the areas before it are

  for (int i = threadIdx.x; i < BNN_EXP_TAB_SIZE; i += blockDim.x) tab[i] = p.exp_tab[i];
  for (int i = threadIdx.x; i < n_cnt; i += blockDim.x) cnt[i] = 0;
  for (int i = threadIdx.x; i < p.sp.prog_len; i += blockDim.x) prog[i] = p.sp.prog[i];

  const long long n_tiles32 = (p.n_tiles16 + 1) >> 1;
  const long long n_pad = p.n_tiles16 * 16;
  const long long t0 = n_tiles32 * blockIdx.x / gridDim.x, t1 = n_tiles32 * (blockIdx.x + 1) / gridDim.x;
  const double* bufl = tile + lane;
  const int nc1 = p.sp.pair_nc1;
  const int stride = 2 * SP_HDR + ((nc1 + 3) & ~3) + ((NR1 + 3) & ~3);          // two padded items per pair
  const int gthreads = GW * 32, gtid = wi * 32 + lane;
  auto group_sync = [&]() { asm volatile("bar.sync %0, %1;" ::"r"(1 + grp), "r"(gthreads) : "memory"); };

  for (int c0 = 0; c0 < p.C; c0 += G) {
    const int gc = min(G, p.C - c0);                          // chains of this group
    const int n_sub = (gc + NCH - 1) / NCH;                   // chain subsets of NCH
    __syncthreads();                                           // previous group's readers are done
    for (int i = threadIdx.x; i < gc * p.sp.wlen; i += blockDim.x) {
      const int c = i / p.sp.wlen, j = i - c * p.sp.wlen;
      const int idx = __ldg(p.sp.widx + j);
      wsm[i] = idx < 0 ? 0.0 : __ldg(p.wp + (long long)(c0 + c) * g.PB + idx);
    }
    __syncthreads();
    if (grp >= n_groups) continue;                             // (left-over warps when nwarps is not a multiple of GW)
    for (long long w32 = t0 + grp; w32 < t1; w32 += n_groups) {
      // X tile -> [feature][row], loaded by the whole group; global reads are contiguous (32 * F_pad doubles)
      const double* xt = p.x + w32 * 32 * (long long)g.F_pad;
      group_sync();                                            // the previous tile's readers are done
      for (int e0 = gtid; e0 < 32 * g.F_pad; e0 += 4 * gthreads) {
        double v[4];
#pragma unroll
        for (int uu = 0; uu < 4; ++uu) {
          const int idx = e0 + uu * gthreads;
          v[uu] = (idx < 32 * g.F_pad && w32 * 32 + idx / g.F_pad < n_pad) ? __ldg(xt + idx) : 0.0;
        }
#pragma unroll
        for (int uu = 0; uu < 4; ++uu) {
          const int idx = e0 + uu * gthreads;
          const int r = idx / g.F_pad, cp = idx - r * g.F_pad;
          const int cidx = cp ^ ((r & 1) * g.x_swz);
          if (idx < 32 * g.F_pad && cidx < g.F) tile[cidx * SP_US + r] = v[uu];
        }
      }
      group_sync();
      for (int sub = wi; sub < n_sub; sub += GW) {
        int ch[NCH];
        const double* w[NCH];
        double out[NCH][SP_MAX_O];
        double alpha1[NCH], alpha2[NCH];
#pragma unroll
        for (int q = 0; q < NCH; ++q) {
          ch[q] = min(NCH * sub + q, gc - 1);
          w[q] = wsm + (size_t)ch[q] * p.sp.wlen;
#pragma unroll
          for (int o = 0; o < SP_MAX_O; ++o) out[q][o] = w[q][o];
          w[q] += SP_MAX_O;
          alpha1[q] = (ACT == BNN_ACT_LEAKY && p.alpha) ? p.alpha[(c0 + ch[q]) * g.L + 0] : 0.0;
          alpha2[q] = (ACT == BNN_ACT_LEAKY && p.alpha) ? p.alpha[(c0 + ch[q]) * g.L + 1] : 0.0;
        }
        const int* it = prog;
        for (int n = 0; n < p.sp.n_items; n += 2, it += stride)
          sparse_pair<ACT, NCH, NR1, NR2, NC1>(it, nc1, O, w, bufl, alpha1, alpha2, tab, out);
#pragma unroll
        for (int q = 0; q < NCH; ++q) {
          if (NCH * sub + q < gc) {
            __syncwarp();
#pragma unroll
            for (int o = 0; o < SP_MAX_O; ++o) zs[lane * ZS + o] = out[q][o];
            __syncwarp();
            bnn_epilogue<false, true>(p, c0 + ch[q], w32 * 2, lane, zs, ZS, tab, cnt, nullptr, nullptr);
          }
        }
      }
    }
  }
  if (n_cnt) {
    __syncthreads();
    for (int i = threadIdx.x; i < n_cnt; i += blockDim.x)
      if (cnt[i]) atomicAdd(&p.counts[i], cnt[i]);
  }
}

// =============================================================================================
// host side: shared-memory plans, program builder, launchers
// =============================================================================================
// shared-memory plan of k_fwd_sparse: chains per unit, chains per resident weight group and warps per CTA
static size_t sparse_fixed_bytes(const NetGeom& g, const SparseParams& sp, int C) {
  return BNN_EXP_TAB_SIZE * sizeof(double) + (size_t)bnn_smem_counts(g, C) * sizeof(int) +
         (size_t)(sp.prog_len + 8) * sizeof(int) + 16;
}
static size_t sparse_warp_bytes(const NetGeom& g, const SparseParams& sp, int nch) {
  return ((size_t)(g.F + nch * sp.slots) * SP_US + 32 * (SP_MAX_O + 1)) * sizeof(double);
}
static bool sparse_plan(const NetGeom& g, const SparseParams& sp, int C, int nch, int* group, int* nwarps) {
  const size_t cap = BNN_MAX_DYN_SMEM;
  const size_t fixed = sparse_fixed_bytes(g, sp, C), per_warp = sparse_warp_bytes(g, sp, nch);
  const size_t per_chain = (size_t)sp.wlen * sizeof(double);
  const int c_up = (C + nch - 1) / nch * nch;
  const int max_warps = (nch == 4) ? 10 : 16;
  // Warps first: the kernel is latency-bound (two to three warps per scheduler), and a smaller resident chain group
  // only costs another sweep over the tiles (X comes from L2 / HBM at a few percent of the step).  The rest of the
  // shared memory then takes as many chains' weight streams as fit.
  for (int w = max_warps; w >= 1; --w) {
    if (fixed + (size_t)w * per_warp + nch * per_chain > cap) continue;
    size_t gr = (cap - fixed - (size_t)w * per_warp) / per_chain;
    gr = gr / nch * nch;
    if (gr > (size_t)c_up) gr = c_up;
    *group = (int)gr;
    *nwarps = w;
    return true;
  }
  return false;
}

constexpr int SPARSE_PAIR_NCH = 2;      // chains a thread of k_fwd_pairs evaluates together
// dynamic shared memory of k_fwd_pairs: `group` resident chains, `nwarps` warps that share one X tile per `share`
static size_t pairs_bytes(const FwdParams& p, int group, int share, int nwarps) {
  const size_t n_cnt = bnn_smem_counts(p.g, p.C);
  return BNN_EXP_TAB_SIZE * sizeof(double) + (((n_cnt + 3) & ~(size_t)3) + p.sp.prog_len + 4) * sizeof(int) +
         (size_t)group * p.sp.wlen * sizeof(double) + (size_t)(nwarps / share) * p.g.F * SP_US * sizeof(double) +
         (size_t)nwarps * 32 * (SP_MAX_O + 1) * sizeof(double);
}
// shared-memory plan of k_fwd_pairs: resident chains, warps per group, warps
static bool pairs_plan(const FwdParams& p, int nch, int* group, int* share, int* nwarps, size_t* bytes) {
  const int max_warps = (nch == 1) ? 24 : 16;
  const int c_up = (p.C + nch - 1) / nch * nch;
  // all chains resident if they fit next to a useful number of warps, else as many as fit with the full set of warps
  for (int gch = c_up; gch >= nch; gch -= nch) {
    const int n_sub = gch / nch;
    int gw = n_sub < 8 ? n_sub : 8;
    while (max_warps % gw) --gw;                       // groups tile the CTA exactly
    for (int w = max_warps; w >= gw; w -= gw) {
      const size_t need = pairs_bytes(p, gch, gw, w);
      if (need <= BNN_MAX_DYN_SMEM && (w >= max_warps / 2 || gch == nch)) {
        *group = gch; *share = gw; *nwarps = w; *bytes = need;
        return true;
      }
    }
  }
  return false;
}

// The (units, units) shapes of uniform block pairs with a compiled instantiation of k_fwd_pairs: calls
// f(PairShape<NR1, NR2>{}) for the one equal to (nr1, nr2) and returns whether there is one.
template <int NR1, int NR2>
struct PairShape { static constexpr int nr1 = NR1, nr2 = NR2; };
template <typename F>
static bool with_pair_shape(int nr1, int nr2, F&& f) {
  auto is = [&](auto s) { return decltype(s)::nr1 == nr1 && decltype(s)::nr2 == nr2 && (f(s), true); };
  return is(PairShape<3, 2>{}) || is(PairShape<2, 1>{}) || is(PairShape<2, 2>{}) || is(PairShape<4, 2>{});
}

// The dataflow program of a block-masked network (format above).
// Per hidden layer, consecutive rows whose kept columns span the same range [c0, c0+nc) form a block
// (create_mask, BNN_lib.py:16-47 produces exactly such blocks); blocks are cut into items of at most 4 rows.
// Columns inside the range that the mask drops are harmless (their weights are exactly zero).  Items are
// emitted in dependency order starting from the last hidden layer, each unit of an earlier layer gets a
// scratch slot that is released after its last reader.  The output layer is evaluated densely.
namespace {
struct SpItem { int l, r0, nr, c0, nc; };
}
bool bnn_sparse_build(const NetGeom& g, const double* mask, SparseProgram* out) {
  std::vector<int>& prog = out->prog;
  std::vector<int>& widx = out->widx;
  SparseParams& sp = out->sp;
  prog.clear();
  widx.clear();
  sp = SparseParams{};
  if (g.L < 2 || g.O > SP_MAX_O) return false;
  const int H = g.L - 1;                        // hidden layers
  const LayerGeom& lo = g.l[H];
  const int op = (lo.out + 1) & ~1;
  std::vector<std::vector<SpItem>> items(H);
  std::vector<std::vector<int>> unit_item(H), readers(H), slot(H);
  long long n_fma = 0, dense = 0;
  for (int l = 0; l < g.L; ++l) dense += (long long)g.l[l].out * g.l[l].in;
  for (int l = 0; l < H; ++l) {
    const LayerGeom& lg = g.l[l];
    const int cols = lg.in + lg.bias;
    auto range_of = [&](int row, int& c0, int& nc) {
      int lo_ = -1, hi = -1;
      for (int k = 0; k < lg.in; ++k)
        if (mask[lg.c_off + row * cols + lg.bias + k] != 0.0) { if (lo_ < 0) lo_ = k; hi = k; }
      c0 = lo_ < 0 ? 0 : lo_;
      nc = lo_ < 0 ? 0 : hi - lo_ + 1;
    };
    unit_item[l].assign(lg.out, -1);
    readers[l].assign(lg.out, 0);
    slot[l].assign(lg.out, -1);
    int r = 0;
    while (r < lg.out) {
      int c0, nc;
      range_of(r, c0, nc);
      int r1 = r + 1;
      while (r1 < lg.out) {
        int d0, dn;
        range_of(r1, d0, dn);
        if (d0 != c0 || dn != nc) break;
        ++r1;
      }
      for (int q = r; q < r1; q += 4) {
        const int nr = (r1 - q < 4) ? r1 - q : 4;
        for (int i = 0; i < nr; ++i) unit_item[l][q + i] = (int)items[l].size();
        items[l].push_back({l, q, nr, c0, nc});
        n_fma += (long long)nr * nc;
      }
      r = r1;
    }
    if (l > 0)
      for (const SpItem& it : items[l])
        for (int k = 0; k < it.nc; ++k) readers[l - 1][it.c0 + k]++;
  }
  n_fma += (long long)lo.out * lo.in;
  if (n_fma * 4 > dense) return false;          // the cover is not worth it (more than a quarter of the dense work)

  // weight stream starts with the output-layer bias (SP_MAX_O entries)
  for (int o = 0; o < SP_MAX_O; ++o) widx.push_back(o < lo.out ? lo.b_off + o : -1);

  std::vector<std::vector<char>> done(H);
  for (int l = 0; l < H; ++l) done[l].assign(items[l].size(), 0);
  std::vector<SpItem> order;                    // the items in program order
  std::vector<int> free_slots;                  // released slots, reused lowest first
  int n_slots = 0;
  auto take_slot = [&]() {
    if (free_slots.empty()) return n_slots++;
    size_t best = 0;
    for (size_t i = 1; i < free_slots.size(); ++i) if (free_slots[i] < free_slots[best]) best = i;
    int v = free_slots[best];
    free_slots.erase(free_slots.begin() + best);
    return v;
  };
  // explicit stack instead of recursion: (layer, item, next column to check)
  struct Frame { int l, idx, k; };
  for (size_t top = 0; top < items[H - 1].size(); ++top) {
    std::vector<Frame> st{{H - 1, (int)top, 0}};
    while (!st.empty()) {
      Frame& f = st.back();
      const SpItem it = items[f.l][f.idx];
      if (done[f.l][f.idx]) { st.pop_back(); continue; }
      bool pushed = false;
      if (f.l > 0) {
        for (; f.k < it.nc; ++f.k) {
          const int prod = unit_item[f.l - 1][it.c0 + f.k];
          if (!done[f.l - 1][prod]) { st.push_back({f.l - 1, prod, 0}); pushed = true; break; }
        }
      }
      if (pushed) continue;
      // emit the item: program entry ...
      const int l = f.l, idx = f.idx;
      const LayerGeom& lg = g.l[l];
      const bool to_out = (l == H - 1);
      prog.push_back(l | (it.nr << 8) | (to_out ? (1 << 16) : 0));
      prog.push_back(it.nc);
      prog.push_back(l > 0 ? 1 : 0);
      prog.push_back(0);
      for (int i = 0; i < 4; ++i) {
        int off = 0;
        if (!to_out && i < it.nr) {
          const int s = take_slot();
          slot[l][it.r0 + i] = s;
          off = (g.F + s) * SP_US;
        }
        prog.push_back(off);
      }
      for (int k = 0; k < it.nc; ++k)
        prog.push_back(l == 0 ? (it.c0 + k) * SP_US : (g.F + slot[l - 1][it.c0 + k]) * SP_US);
      while (prog.size() % 4) prog.push_back(0);
      // ... and its weights in consumption order
      const int nrp = (it.nr + 1) & ~1;
      for (int i = 0; i < nrp; ++i) widx.push_back(i < it.nr ? lg.b_off + it.r0 + i : -1);
      for (int k = 0; k < it.nc; ++k)
        for (int i = 0; i < nrp; ++i) {
          const int r = it.r0 + i, cc = it.c0 + k;
          widx.push_back(i < it.nr ? lg.w_off + r * lg.stride + (cc ^ ((r & 1) * lg.swz)) : -1);
        }
      if (to_out)
        for (int i = 0; i < it.nr; ++i)
          for (int o = 0; o < op; ++o) {
            const int u = it.r0 + i;
            widx.push_back(o < lo.out ? lo.w_off + o * lo.stride + (u ^ ((o & 1) * lo.swz)) : -1);
          }
      if (l > 0)
        for (int k = 0; k < it.nc; ++k)
          if (--readers[l - 1][it.c0 + k] == 0) free_slots.push_back(slot[l - 1][it.c0 + k]);
      done[l][idx] = 1;
      order.push_back(it);
      st.pop_back();
    }
  }
  sp.prog_len = (int)prog.size();
  sp.n_items = (int)order.size();
  sp.wlen = (int)widx.size();
  sp.slots = n_slots < 1 ? 1 : n_slots;
  // Uniform block pairs: two hidden layers, and the program is (first-layer item a, the second-layer item b that reads
  // exactly a's units) repeated with one shape that k_fwd_pairs is compiled for -- then the hidden units stay in
  // registers.  b reads a's units when it reads as many units as a makes, starting at a's first.
  if (H == 2 && order.size() >= 2 && order.size() % 2 == 0) {
    const SpItem a0 = order[0], b0 = order[1];
    bool uniform = a0.nc > 0 && with_pair_shape(a0.nr, b0.nr, [](auto) {});
    for (size_t n = 0; n < order.size() && uniform; n += 2) {
      const SpItem &a = order[n], &b = order[n + 1];
      uniform = a.l == 0 && b.l == 1 && b.c0 == a.r0 && b.nc == a.nr && a.nc == a0.nc && a.nr == a0.nr && b.nr == b0.nr;
    }
    if (uniform) { sp.pair_nc1 = a0.nc; sp.pair_nr1 = a0.nr; sp.pair_nr2 = b0.nr; }
  }
  // the largest pass must fit the interpreter's shared memory with two chains per unit
  int group, nwarps;
  return sparse_plan(g, sp, BNN_MAX_SETS_PER_PASS, 2, &group, &nwarps);
}

template <int ACT, int NCH>
static cudaError_t launch_sparse_n(const FwdParams& p0, int n_sms, cudaStream_t st) {
  auto kern = k_fwd_sparse<ACT, NCH>;
  FwdParams p = p0;
  int group = 0, nwarps = 0;
  if (!sparse_plan(p.g, p.sp, p.C, NCH, &group, &nwarps)) return cudaErrorInvalidConfiguration;
  p.sp.group = group;
  const long long n_tiles32 = (p.n_tiles16 + 1) >> 1;
  int grid = (int)(n_tiles32 < n_sms ? n_tiles32 : n_sms);
  // small problems: no more warps than units per CTA
  const long long units = ((n_tiles32 + grid - 1) / grid) * ((group + NCH - 1) / NCH);
  if (units < nwarps) nwarps = (int)units;
  const size_t bytes = sparse_fixed_bytes(p.g, p.sp, p.C) + (size_t)group * p.sp.wlen * sizeof(double) +
                       (size_t)nwarps * sparse_warp_bytes(p.g, p.sp, NCH);
  if (cudaError_t e = bnn_prepare_kernel((const void*)kern, BNN_MAX_DYN_SMEM)) return e;
  kern<<<grid, nwarps * 32, bytes, st>>>(p);
  return cudaGetLastError();
}

template <int ACT, int NR1, int NR2, int NC1 = 0>
static cudaError_t launch_pairs(const FwdParams& p0, int n_sms, cudaStream_t st) {
  if (NC1 == 0 && p0.sp.pair_nc1 == 1) return launch_pairs<ACT, NR1, NR2, 1>(p0, n_sms, st);
  auto kern = k_fwd_pairs<ACT, SPARSE_PAIR_NCH, NR1, NR2, NC1>;
  FwdParams p = p0;
  int group = 0, share = 1, nwarps = 0;
  size_t bytes = 0;
  if (!pairs_plan(p, SPARSE_PAIR_NCH, &group, &share, &nwarps, &bytes)) return cudaErrorInvalidConfiguration;
  p.sp.group = group;
  p.sp.share = share;
  const long long n_tiles32 = (p.n_tiles16 + 1) >> 1;
  int grid = (int)(n_tiles32 < n_sms ? n_tiles32 : n_sms);
  // small problems: no more groups than tiles per CTA
  const long long tiles_per_cta = (n_tiles32 + grid - 1) / grid;
  if (tiles_per_cta * share < nwarps) {
    nwarps = (int)tiles_per_cta * share;
    bytes = pairs_bytes(p, group, share, nwarps);
  }
  if (cudaError_t e = bnn_prepare_kernel((const void*)kern, BNN_MAX_DYN_SMEM)) return e;
  kern<<<grid, nwarps * 32, bytes, st>>>(p);
  return cudaGetLastError();
}

template <int ACT>
static cudaError_t launch_sparse_t(const FwdParams& p, int n_sms, cudaStream_t st, const char** which) {
  int group, share, nwarps;
  size_t bytes;
  if (p.C >= 2 && p.sp.pair_nc1 && pairs_plan(p, SPARSE_PAIR_NCH, &group, &share, &nwarps, &bytes)) {
    // uniform block pairs (create_mask with equal node counts per feature group): fused, register-resident path
    if (which) *which = "k_fwd_sparse<pairs>";
    cudaError_t e = cudaErrorInvalidConfiguration;
    with_pair_shape(p.sp.pair_nr1, p.sp.pair_nr2, [&](auto s) {
      e = launch_pairs<ACT, decltype(s)::nr1, decltype(s)::nr2>(p, n_sms, st);
    });
    return e;
  }
  if (which) *which = "k_fwd_sparse";
  if (p.C >= 3 && sparse_plan(p.g, p.sp, p.C, 4, &group, &nwarps)) return launch_sparse_n<ACT, 4>(p, n_sms, st);
  return launch_sparse_n<ACT, 2>(p, n_sms, st);
}

cudaError_t bnn_launch_sparse(const FwdParams& p, int n_sms, cudaStream_t st, const char** which) {
  return bnn_with_act(p.g.act, [&](auto a) { return launch_sparse_t<decltype(a)::value>(p, n_sms, st, which); });
}
