// topk_kernel.cuh -- cosine scoring of query embeddings against the whole entity table with a fused candidate filter:
//
//   pred_norm = F.normalize(pred, dim=-1); entity_norm = F.normalize(node_emb, dim=-1)
//   similarities = pred_norm @ entity_norm.T;  top_scores, top_indices = similarities.topk(k, dim=1)
//                                               (pro_b_gan_infer.py:146-151, :231-236)
//
// The [B, N] similarity matrix (1 GiB at B = 4096, N = 65536) never exists.  Steps (E = 128, k <= 16):
//   1. prepare : row norms; bf16 copies of the normalised table / queries, zero padded to 256 rows        (HBM-bound)
//   2. sample  : bf16 tensor-core scores (CTA pairs, tcgen05.mma.cta_group::2, M = 256 queries x N = 256 entities per
//                MMA group, K = E = 128; query tile stationary, entity tiles streamed by TMA) of every 4th entity (k <= 16; every 2nd above)
//                tile.  Epilogue per query row (one thread each): the maximum of every 32 scores as a packed
//                (score | position) integer key -- one LOP3 per score and a three-input max tree -- pushed through a
//                16-deep sorted insert once per 32 scores.  A small kernel merges a row's lists: tau[row] = the k-th
//                best sampled score, i.e. at least k entities score >= tau.
//   3. scan    : the same MMA pipeline over ALL entity tiles; the matrix goes TMEM -> registers -> compare only.  Per
//                score: one compare with tau and one bit into a 32-bit mask -- no vote, no branch per score; per 32
//                scores a mask that is not empty is appended with its group number to a thread-private list in global memory
//                (about k * 8 / lists entries per list).
//   4. rescore : exact fp32 cosine of every entity whose bit is set, top-k among them (ties: lower index first), and
//                a proof obligation per row: the k-th exact score must beat tau by more than the bf16 error bound --
//                everything that was not a candidate has a bf16 score <= tau -- else the row is flagged and re-done
//                by an exact scan of the table (rare).
// so the returned indices are those of an exact fp32 evaluation, not of the bf16 scores.
// Other shapes (k > 64, E != 128, small tables): exact fp32 scores of a chunk of rows by the SIMT GEMM of the parity
// mode, then one selection CTA per row (topk_select_kernel below; pbg.cu: topk_general).
#pragma once
#include <cuda.h>
#include "ptx.cuh"
#include "tc_common.cuh"
#include "pass_common.cuh"

namespace pbg {

constexpr int kTkStages = 4;          // entity tiles in flight per CTA (32 KB each: 128 entities x 128 dims bf16)
constexpr int kTkCand = 256;          // (group, mask) entries kept per (row, entity range, column half), in global memory
constexpr int kTkMaxRanges = 16;
constexpr int kTkMaxK = 64;           // largest k of the filter path; above it the general path runs
// every stride-th 256-entity tile is sampled for the cut-off.  About stride * k entities (+ those inside the error margin)
// pass it and are rescored -- one 512-byte row read each, the largest part of a call -- while the sample launch costs
// 1 / stride of the scan: measured at B = 4096, N = 65536: k = 10 156 / 141 / 141 us at 1 in 8 / 4 / 2, k = 17 172 / 163 us
// and k = 40 267 / 238 us at 1 in 4 / 2
inline int tk_sample_stride(int k) { return k <= 16 ? 4 : 2; }
constexpr int kTkKeys = 16;           // best group keys a thread keeps per sample list; a row's lists together hold >= 2 k keys (pbg.cu: chunk size)
constexpr int kTkRescoreMax = 1024;   // candidates per row the rescoring kernel takes (about 8 k + a dozen arrive); more: exact scan
constexpr int kTkRescoreWarps = 4;    // rows per rescoring CTA (32 KB of candidate scores / indices in shared memory)
// |bf16 score - exact score| for unit vectors q, t and their bf16 copies q', t' (round to nearest, 8 significant bits:
// relative error up to 2^-8 per entry, so a fixed constant would have to be (2^-7 + 2^-16) * sum |q_i t_i| <= 0.0079):
//   |q'.t' - q.t| <= ||q' - q|| * ||t'|| + ||q|| * ||t' - t|| <= e_q (1 + e_t) + e_t
// with e_q = ||q' - q|| of the query row (measured by topk_tau_kernel) and e_t the largest ||t' - t|| of the table
// (measured by topk_prepare_kernel); + fp32 accumulation of 128 products in the tensor cores and in the rescoring
// (<= 1.5e-5) + the sample keys' 5 truncated mantissa bits (<= 4e-6).  Random rows give e_q ~ 0.0017, e_t ~ 0.0023
// (err ~ 0.0040); rows whose entries all sit just past a power of two reach 2^-8 * ||x|| and err ~ 0.0078.
constexpr float kTkErrSlack = 2e-5f;
__device__ __forceinline__ float tk_err(float e_q, const unsigned* err_t) {
  const float e_t = __uint_as_float(*err_t);
  return e_q * (1.f + e_t) + e_t + kTkErrSlack;
}
enum : int { TK_SAMPLE = 0, TK_SCAN = 1 };

struct alignas(64) TopkParams {
  CUtensorMap tm_q;      // normalised queries bf16 [Bpad, 128]: box 64 x 128 rows
  CUtensorMap tm_t;      // normalised table   bf16 [Npad, 128]: box 64 x 128 rows (one CTA's half of a 256-entity tile)
  int n_rb;              // 256-row query blocks
  int n_tiles;           // visited tiles per query block: every tile (scan) or every tile_stride-th (sample)
  int tile_stride;       // table tile = visited tile * tile_stride
  int total;             // work units = n_rb * n_tiles (one unit = one query block x one visited tile), query-block major
  int span;              // units per CTA pair: pair p takes units [p * span, (p + 1) * span) -- whole device, equal shares
  int n_ranges;          // list slots per (row, column half): the most pairs whose spans meet one query block
  long long N;           // valid entities
  int* samp_keys;        // sample: [Bpad][n_ranges * 2][kTkKeys] best group keys, descending (unused slots: zero)
  const float* tau;      // scan:   [Bpad] cut-off per query row
  unsigned* cand_grp;    // scan:   [Bpad][n_ranges * 2][kTkCand] 32-entity group numbers ...
  unsigned* cand_mask;   //         ... and which of the group's entities scored above tau
  int* cand_cnt;         // scan:   [Bpad][n_ranges * 2] groups found (more than kTkCand: the list overflowed; unused slots: 0)
};

// A pair's span of work units, cut at query-block boundaries: segment = (query block, visited tiles [t0, t1), list slot).
// The slot numbers the pairs that meet a query block in order, so every (row, slot) list has exactly one writer.
struct TkSeg { int rb, t0, t1, slot; };
__device__ __forceinline__ bool tk_next_seg(const TopkParams& p, int pair, int& u, TkSeg& s) {
  const int end = min((pair + 1) * p.span, p.total);
  if (u >= end) return false;
  s.rb = u / p.n_tiles;
  s.t0 = u - s.rb * p.n_tiles;
  s.t1 = min(p.n_tiles, s.t0 + (end - u));
  s.slot = pair - (s.rb * p.n_tiles) / p.span;
  u += s.t1 - s.t0;
  return true;
}

struct TkSmem {
  static constexpr int kQ = 2 * 128 * kBlockK * 2;        // this CTA's 128 query rows, 2 k-blocks; TWO such buffers: the next
                                                          // segment's query tile lands while this segment's tiles stream
  static constexpr int kT = 2 * 128 * kBlockK * 2;        // this CTA's 128 entities of a tile, 2 k-blocks
  static constexpr int kStageOff = 2 * kQ;
  static constexpr int kBarOff = kStageOff + kTkStages * kT;
  static constexpr int kTotal = kBarOff + 256 + 1024;
};
static_assert(TkSmem::kTotal <= 232448, "topk: shared memory budget");

// Programmatic dependent launch along the chain prepare -> sample -> cut-off -> scan -> rescore -> exact scan (pbg.cu says
// which links use it): a kernel releases its successor when it is done with its own work (released at entry, the
// successor's CTAs sat in griddepcontrol.wait beside this kernel's and slowed it), and EVERY thread of every kernel
// waits for its predecessor -- all of it, memory included -- before it touches anything the chain produced; a CTA that
// skipped the wait could let its grid finish, and release the grid after it, too early.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ------------------------------------------------------------------------------------------------ 1. prepare
// One warp per row: inv = 1 / max(||x||, 1e-12) (F.normalize's eps), bf16(x * inv) into a [rows_pad, E] matrix whose
// padding rows are zero.  HBM-bound (E fp32 in, E bf16 + 4 B out per row): a warp takes R rows per iteration, every
// load of those rows in flight before the first reduction (bytes in flight per SM, not instruction count, set the rate),
// and keeps the values in registers for the scaling pass.  <R = 8, V = 1>: E <= 128; <R = 2, V = 4>: E <= 512 in
// registers, wider rows are read a second time.  ERR (the table): the largest row rounding error ||bf16(x * inv) -
// x * inv||_2 (the error bound above) goes to *err_max -- non-negative floats order like their bits, the caller zeroes
// the word.  The queries' errors are measured by topk_tau_kernel, off this kernel's critical path.
__device__ __forceinline__ float tk_store_bf16(__nv_bfloat16* dst, float4 v) {   // returns the squared rounding error
  const __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
  const float2 rl = __bfloat1622float2(lo), rh = __bfloat1622float2(hi);
  uint2 w;
  w.x = *reinterpret_cast<const uint32_t*>(&lo);
  w.y = *reinterpret_cast<const uint32_t*>(&hi);
  *reinterpret_cast<uint2*>(dst) = w;
  const float a = v.x - rl.x, b = v.y - rl.y, c = v.z - rh.x, d = v.w - rh.y;   // exact: x minus its rounding
  return a * a + b * b + c * c + d * d;
}

template <int R, int V, bool ERR>
__global__ void __launch_bounds__(256) topk_prepare_kernel(const float* __restrict__ x, long long rows, long long rows_pad, int E,
                                                           __nv_bfloat16* __restrict__ xn, float* __restrict__ inv,
                                                           unsigned* __restrict__ err_max) {
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const long long warp0 = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const long long nwarp = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
  const bool in_regs = E <= 128 * V;
  float emax = 0.f;   // ERR: this warp's largest row error
  for (long long r0 = warp0 * R; r0 < rows_pad; r0 += nwarp * R) {
    float es[R];
    float4 v[R][V];
    float ss[R];
#pragma unroll
    for (int i = 0; i < R; ++i) {
      ss[i] = 0.f;
      const long long r = r0 + i;
#pragma unroll
      for (int j = 0; j < V; ++j) {
        const int c = lane * 4 + j * 128;
        v[i][j] = (r < rows && c < E && in_regs) ? *reinterpret_cast<const float4*>(x + r * E + c) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
#pragma unroll
    for (int i = 0; i < R; ++i) {
      const long long r = r0 + i;
      if (in_regs) {
#pragma unroll
        for (int j = 0; j < V; ++j) ss[i] += v[i][j].x * v[i][j].x + v[i][j].y * v[i][j].y + v[i][j].z * v[i][j].z + v[i][j].w * v[i][j].w;
      } else if (r < rows) {
        for (int c = lane * 4; c < E; c += 128) {
          const float4 w = *reinterpret_cast<const float4*>(x + r * E + c);
          ss[i] += w.x * w.x + w.y * w.y + w.z * w.z + w.w * w.w;
        }
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
      for (int i = 0; i < R; ++i) ss[i] += __shfl_xor_sync(0xffffffffu, ss[i], o);
    }
#pragma unroll
    for (int i = 0; i < R; ++i) {
      const long long r = r0 + i;
      es[i] = 0.f;
      if (r >= rows_pad) continue;
      if (r >= rows) {
        for (int c = lane * 4; c < E; c += 128) store4<__nv_bfloat16>(xn + r * E + c, make_float4(0.f, 0.f, 0.f, 0.f));
        continue;
      }
      const float iv = 1.f / fmaxf(sqrtf(ss[i]), 1e-12f);
      if (lane == 0) inv[r] = iv;
      if (in_regs) {
#pragma unroll
        for (int j = 0; j < V; ++j) {
          const int c = lane * 4 + j * 128;
          const float4 y = make_float4(v[i][j].x * iv, v[i][j].y * iv, v[i][j].z * iv, v[i][j].w * iv);
          if (c < E) { if (ERR) es[i] += tk_store_bf16(xn + r * E + c, y); else store4<__nv_bfloat16>(xn + r * E + c, y); }
        }
      } else {
        for (int c = lane * 4; c < E; c += 128) {
          const float4 w = *reinterpret_cast<const float4*>(x + r * E + c);
          const float4 y = make_float4(w.x * iv, w.y * iv, w.z * iv, w.w * iv);
          if (ERR) es[i] += tk_store_bf16(xn + r * E + c, y); else store4<__nv_bfloat16>(xn + r * E + c, y);
        }
      }
    }
    if (ERR) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int i = 0; i < R; ++i) es[i] += __shfl_xor_sync(0xffffffffu, es[i], o);
      }
#pragma unroll
      for (int i = 0; i < R; ++i) emax = fmaxf(emax, sqrtf(es[i]));
    }
  }
  if (ERR && lane == 0 && emax > 0.f) atomicMax(err_max, __float_as_uint(emax));
  pdl_launch_dependents();   // at the END: successors released at entry sit beside this kernel's blocks and slow them
}

// ------------------------------------------------------------------------------------------------ 2 / 3. sample, scan
// MODE TK_SAMPLE: visited tiles are every tile_stride-th tile; per (row, range, column half) the kTkKeys best group
//                 keys go to samp_keys.  MODE TK_SCAN: every tile; (group, mask) candidate lists.
// (score bits with the low 5 bits replaced by the position) as ONE lop3: (a & b) | c
__device__ __forceinline__ int tk_key(uint32_t bits, int j) {
  int d;
  asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=r"(d) : "r"(bits), "r"(0xFFFFFFE0u), "r"(j));
  return d;
}

template <int MODE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kPassThreads, 1)
pbg_topk_scan_kernel(const __grid_constant__ TopkParams p) {
  using L = TkSmem;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::kBarOff);
  uint64_t* empty_bar = full_bar + kTkStages;
  uint64_t* tmem_full = empty_bar + kTkStages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint64_t* q_full = tmem_empty + 2;     // [2]
  uint64_t* q_empty = q_full + 2;        // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(q_empty + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int pair = static_cast<int>(blockIdx.x) >> 1;

  if (threadIdx.x == 0) {
    prefetch_tmap(&p.tm_q);
    prefetch_tmap(&p.tm_t);
    for (int s = 0; s < kTkStages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&tmem_full[s], 1); mbar_init(&tmem_empty[s], 2 * kEpiWarps); }
    for (int s = 0; s < 2; ++s) { mbar_init(&q_full[s], 1); mbar_init(&q_empty[s], 1); }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc_pair<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t lead_tmem_empty = mapa_u32(smem_u32(tmem_empty), 0);
  pdl_wait();   // the prologue above touched nothing of the chain; the queries, the cut-offs, the lists do

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer (both CTAs, their halves)
    if (lane == 0) {
      const uint32_t lead_full = mapa_u32(smem_u32(full_bar), 0);
      const uint32_t lead_q_full = mapa_u32(smem_u32(q_full), 0);
      uint32_t stage = 0, phase = 0, nseg = 0;
      int u = pair * p.span;
      TkSeg sg;
      while (tk_next_seg(p, pair, u, sg)) {
        const int rb = sg.rb;
        // the query tile of this segment into buffer nseg & 1 (free once the MMAs of segment nseg - 2 are done: this
        // thread runs a ring ahead of the MMAs, so the tile is in flight while the previous segment still computes)
        const uint32_t qb = nseg & 1, qphase = (nseg >> 1) & 1;
        mbar_wait(&q_empty[qb], qphase ^ 1);
        if (leader) mbar_arrive_expect_tx(&q_full[qb], 2u * L::kQ);
        for (int kb = 0; kb < 2; ++kb)
          tma_load_2d_pair(smem + qb * L::kQ + kb * (L::kQ / 2), &p.tm_q, lead_q_full + qb * 8, kb * kBlockK, rb * 256 + static_cast<int>(rank) * 128);
        ++nseg;
        for (int t = sg.t0; t < sg.t1; ++t) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          if (leader) mbar_arrive_expect_tx(&full_bar[stage], 2u * L::kT);
          uint8_t* st = smem + L::kStageOff + stage * L::kT;
          for (int kb = 0; kb < 2; ++kb)
            tma_load_2d_pair(st + kb * (L::kT / 2), &p.tm_t, lead_full + stage * 8, kb * kBlockK,
                             t * p.tile_stride * 256 + static_cast<int>(rank) * 128);
          if (++stage == kTkStages) { stage = 0; phase ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer (leader)
    if (leader && lane == 0) {
      constexpr uint32_t idesc = make_idesc_bf16(256, 256);
      uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0, nseg = 0;
      int u = pair * p.span;
      TkSeg sg;
      while (tk_next_seg(p, pair, u, sg)) {
        const uint32_t qb = nseg & 1;
        mbar_wait(&q_full[qb], (nseg >> 1) & 1);
        ++nseg;
        tc_fence_after();
        for (int t = sg.t0; t < sg.t1; ++t) {
          mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + acc * 256;
          const uint32_t sq = smem_u32(smem + qb * L::kQ), stt = smem_u32(smem + L::kStageOff + stage * L::kT);
#pragma unroll
          for (int kb = 0; kb < 2; ++kb) {
            const uint64_t da = make_kmajor_sw128_desc(sq + kb * (L::kQ / 2));
            const uint64_t db = make_kmajor_sw128_desc(stt + kb * (L::kT / 2));
#pragma unroll
            for (int k = 0; k < kBlockK / kUmmaK; ++k) umma_bf16_pair(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
          }
          umma_commit_pair(&empty_bar[stage], 3);
          umma_commit_pair(&tmem_full[acc], 3);
          if (++stage == kTkStages) { stage = 0; phase ^= 1; }
          if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
        umma_commit_pair(&q_empty[qb], 3);   // this query buffer may be overwritten once these MMAs are done
      }
    }
    __syncwarp();
  } else {
    // ------------------------------------------------------------ filter warps (both CTAs): one query row per thread
    const int wep = warp - 2, q = warp & 3, half = wep >> 2;
    uint32_t acc = 0, acc_phase = 0;
    int u = pair * p.span;
    TkSeg sg;
    while (tk_next_seg(p, pair, u, sg)) {
      const int rb = sg.rb, rg = sg.slot;
      const long long row = static_cast<long long>(rb) * 256 + static_cast<int>(rank) * 128 + q * 32 + lane;
      const int t0 = sg.t0, t1 = sg.t1;
      int m[kTkKeys];                       // sample: the best group keys so far, descending
#pragma unroll
      for (int i = 0; i < kTkKeys; ++i) m[i] = 0;
      const float tau = MODE == TK_SCAN ? p.tau[row] : 0.f;
      const long long lbase = row * (p.n_ranges * 2) + rg * 2 + half;
      // scan: the list lives in global memory -- an append is one predicated 8-byte pair of stores every few thousand
      // scores per thread, and its length is then bounded by memory, not by what is left of shared memory
      unsigned* lgrp = MODE == TK_SCAN ? p.cand_grp + lbase * kTkCand : nullptr;
      unsigned* lmsk = MODE == TK_SCAN ? p.cand_mask + lbase * kTkCand : nullptr;
      int cnt = 0;                          // scan: groups appended (may run past kTkCand: overflow)
      for (int t = t0; t < t1; ++t) {
        mbar_wait(&tmem_full[acc], acc_phase);
        tc_fence_after();
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * 256 + half * 128;
        const unsigned grp0 = static_cast<unsigned>(t * p.tile_stride) * 8u + static_cast<unsigned>(half) * 4u;   // 32-entity groups
        uint32_t va[32], vb[32];
        auto process = [&](const uint32_t (&cur)[32], int g) {
          if (MODE == TK_SAMPLE) {
            // positive floats order like integers and negative ones are negative integers: a signed max with a floor
            // of 0 is the float max of the positives; the low 5 bits carry the position (a tie-break, never decoded)
            int a0 = 0, a1 = 0, a2 = 0, a3 = 0;
#pragma unroll
            for (int j = 0; j < 32; j += 8) {
              a0 = __vimax3_s32(a0, tk_key(cur[j + 0], j + 0), tk_key(cur[j + 1], j + 1));
              a1 = __vimax3_s32(a1, tk_key(cur[j + 2], j + 2), tk_key(cur[j + 3], j + 3));
              a2 = __vimax3_s32(a2, tk_key(cur[j + 4], j + 4), tk_key(cur[j + 5], j + 5));
              a3 = __vimax3_s32(a3, tk_key(cur[j + 6], j + 6), tk_key(cur[j + 7], j + 7));
            }
            const int a = max(__vimax3_s32(a0, a1, a2), a3);
            // sorted insert, every level from the old value above it: m_i = max(m_i, min(m_{i-1}, a))
#pragma unroll
            for (int i = kTkKeys - 1; i > 0; --i) m[i] = max(m[i], min(m[i - 1], a));
            m[0] = max(m[0], a);
          } else {
            // two instructions per score: tau - s is negative exactly when s > tau (tau >= 0), and a funnel shift moves
            // that sign bit into the mask; score j ends up at bit 31 - j
            unsigned mask = 0u;
#pragma unroll
            for (int j = 0; j < 32; ++j) mask = __funnelshift_l(__float_as_uint(tau - __uint_as_float(cur[j])), mask, 1);
            if (mask != 0u) {
              if (cnt < kTkCand) { lgrp[cnt] = grp0 + static_cast<unsigned>(g); lmsk[cnt] = mask; }
              ++cnt;
            }
          }
        };
        tmem_ld_32x32_ptr(taddr, va);
#pragma unroll 1
        for (int gp = 0; gp < 2; ++gp) {
          tmem_ld_wait();
          tmem_ld_32x32_ptr(taddr + (2 * gp + 1) * 32, vb);
          process(va, 2 * gp);
          tmem_ld_wait();
          if (gp == 0) {
            tmem_ld_32x32_ptr(taddr + 64, va);
          } else {  // last read of this accumulator stage
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_remote(lead_tmem_empty + acc * 8);
          }
          process(vb, 2 * gp + 1);
        }
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
      if (MODE == TK_SAMPLE) {
#pragma unroll
        for (int i = 0; i < kTkKeys; ++i) p.samp_keys[lbase * kTkKeys + i] = m[i];
      } else {
        p.cand_cnt[lbase] = cnt;
      }
      // the pair that finishes a query block empties the block's list slots that no pair wrote
      if (t1 == p.n_tiles) {
        for (int sl = rg + 1; sl < p.n_ranges; ++sl) {
          const long long lb = row * (p.n_ranges * 2) + sl * 2 + half;
          if (MODE == TK_SAMPLE) {
#pragma unroll
            for (int i = 0; i < kTkKeys; ++i) p.samp_keys[lb * kTkKeys + i] = 0;
          } else {
            p.cand_cnt[lb] = 0;
          }
        }
      }
    }
  }
  // the successor (cut-off / rescoring kernel) may start now, while this CTA tears down: released at entry its CTAs sat
  // in griddepcontrol.wait beside this kernel's for its whole length and slowed it (k = 64, B = 1024: 214 against 170 us)
  pdl_launch_dependents();
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_pair<512>(tmem_base);
  }
}

// One warp per query row: s_k = the k-th largest of the row's sampled group keys (n_lists x kTkKeys of them) with its
// position bits cleared -- at least k sampled entities have a bf16 score >= s_k, hence an exact score >= s_k - err, so
// the k-th exact score of the row is >= s_k - err (err = tk_err of the row).  The scan's cut-off is tau = s_k - 2 err -
// 1e-4: every entity that is NOT marked has a bf16 score <= tau, i.e. an exact score <= tau + err < s_k - err <= the k-th
// exact score -- the proof obligation of the rescoring kernel holds by construction (it is still checked), at the price
// of about a dozen more candidates per row than a cut-off at s_k itself.  Fewer than k positive keys: tau = 0.
// The row's e_q is measured here (E = 128: 4 dimensions per lane) and kept in err_q[row] for the rescoring kernel.
__global__ void __launch_bounds__(256) topk_tau_kernel(const int* __restrict__ samp_keys, int n_lists, long long B, long long rows_pad,
                                                       int k, const float* __restrict__ q, const float* __restrict__ inv_q,
                                                       const __nv_bfloat16* __restrict__ qn, float* __restrict__ err_q,
                                                       const unsigned* __restrict__ err_t, float* __restrict__ tau) {
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const long long row = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  if (row >= rows_pad) return;
  if (row >= B) { if (lane == 0) tau[row] = 0.f; return; }
  const int n = n_lists * kTkKeys;           // <= 32 lists x 16 keys: 16 per lane
  int mine[kTkKeys];
#pragma unroll
  for (int i = 0; i < kTkKeys; ++i) { const int c = i * 32 + lane; mine[i] = c < n ? samp_keys[row * n + c] : 0; }
  float err;
  {  // ||bf16(q^) - q^||, q^ = q * inv_q rounded as the prepare kernel rounded it
    const float4 v = *reinterpret_cast<const float4*>(q + row * 128 + 4 * lane);
    const float iq = inv_q[row];
    const uint2 w = *reinterpret_cast<const uint2*>(qn + row * 128 + 4 * lane);
    const float2 lo = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w.x));
    const float2 hi = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w.y));
    const float a = __fmul_rn(v.x, iq) - lo.x, b = __fmul_rn(v.y, iq) - lo.y, c = __fmul_rn(v.z, iq) - hi.x, d = __fmul_rn(v.w, iq) - hi.y;
    float es = a * a + b * b + c * c + d * d;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) es += __shfl_xor_sync(0xffffffffu, es, o);
    if (lane == 0) err_q[row] = sqrtf(es);
    err = tk_err(sqrtf(es), err_t);
  }
  int kth = 0;
  for (int r = 0; r < k; ++r) {
    int best = 0, at = 0;
#pragma unroll
    for (int i = 0; i < kTkKeys; ++i) if (mine[i] > best) { best = mine[i]; at = i; }
    int wbest = best;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) wbest = max(wbest, __shfl_xor_sync(0xffffffffu, wbest, o));
    // remove one instance of the winner (the lowest lane that holds it)
    const unsigned who = __ballot_sync(0xffffffffu, best == wbest && wbest > 0);
    if (who != 0u && lane == __ffs(who) - 1) {
#pragma unroll
      for (int i = 0; i < kTkKeys; ++i) if (i == at) mine[i] = 0;
    }
    kth = wbest;
  }
  if (lane == 0) tau[row] = kth > 0 ? fmaxf(__int_as_float(kth & ~0x1F) - (2.f * err + 1e-4f), 0.f) : 0.f;
  pdl_launch_dependents();   // (an exited thread counts as well)
}

// ------------------------------------------------------------------------------------------------ 4. rescore
// One warp per query row (E = 128): the candidates are the set bits of the row's (group, mask) lists.  Exact scores,
// the k best (descending; ties: lower index), and the proof that nothing else can belong to them: everything that is
// not a candidate has a bf16 score <= tau.  flag[row] = 1 asks for the exact scan (list overflow, too many or too few
// candidates, proof failed).  Each lane scores one candidate at a time (its whole 128-dim dot, the normalised query
// broadcast from shared memory): 32 candidates and 32 independent row reads in flight per warp, no shuffles.
__global__ void __launch_bounds__(32 * kTkRescoreWarps) topk_rescore_kernel(const float* __restrict__ q, const float* __restrict__ inv_q,
                                                           const float* __restrict__ table, const float* __restrict__ inv_t,
                                                           const unsigned* __restrict__ cand_grp, const unsigned* __restrict__ cand_mask,
                                                           const int* __restrict__ cand_cnt, const float* __restrict__ tau,
                                                           const float* __restrict__ err_q, const unsigned* __restrict__ err_t,
                                                           int n_lists, long long B, long long N, int k,
                                                           long long* __restrict__ out_idx, float* __restrict__ out_score,
                                                           int* __restrict__ flag) {
  __shared__ float es_s[kTkRescoreWarps][kTkRescoreMax];
  __shared__ int ei_s[kTkRescoreWarps][kTkRescoreMax];
  // (no early launch of the successor here: the exact-scan CTAs carry up to 131 KB of shared memory each and, parked on
  // an SM, would take the room of four of this kernel's CTAs -- k = 64 ran 25 % slower that way)
  pdl_wait();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  float* es = es_s[w]; int* ei = ei_s[w];
  const long long row = static_cast<long long>(blockIdx.x) * kTkRescoreWarps + w;
  if (row >= B) return;
  // this lane's four dimensions of the normalised query stay in registers
  float4 qv = *reinterpret_cast<const float4*>(q + row * 128 + 4 * lane);
  {
    const float iq = inv_q[row];
    qv.x *= iq; qv.y *= iq; qv.z *= iq; qv.w *= iq;
  }
  // decode: the row's lists are one flat sequence of (group, mask) entries (list l = lane l's count, a shuffle prefix
  // sum gives every list's offset); 32 entries per round, one per lane, all their loads in flight together; the set
  // bits are compacted into ei[] in (entry, bit) order with a ballot per round -- deterministic, no atomics
  int c_l = lane < n_lists ? cand_cnt[row * n_lists + lane] : 0;
  const bool overflow = __any_sync(0xffffffffu, c_l > kTkCand);
  c_l = min(c_l, kTkCand);
  int pre = c_l;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, pre, o); if (lane >= o) pre += v; }
  const int total = __shfl_sync(0xffffffffu, pre, 31);
  const int start = pre - c_l;
  int ncand = 0;
  for (int i0 = 0; i0 < total; i0 += 32) {
    const int i = i0 + lane;
    int l = 0, st = 0;
    for (int ll = 0; ll < n_lists; ++ll) {
      const int pe = __shfl_sync(0xffffffffu, pre, ll), ps = __shfl_sync(0xffffffffu, start, ll);
      if (i >= ps && i < pe) { l = ll; st = ps; }
    }
    unsigned g = 0u, mk = 0u;
    if (i < total) {
      const long long at = (row * n_lists + l) * kTkCand + (i - st);
      g = cand_grp[at]; mk = cand_mask[at];
    }
    while (__any_sync(0xffffffffu, mk != 0u)) {
      const bool has = mk != 0u;
      const unsigned who = __ballot_sync(0xffffffffu, has);
      if (has) {
        const int b = 31 - __clz(mk);                 // highest bit first = lowest score index j first (bit 31 - j)
        mk &= ~(1u << b);
        const long long ent = static_cast<long long>(g) * 32 + (31 - b);
        const int pos = ncand + __popc(who & ((1u << lane) - 1u));
        if (pos < kTkRescoreMax) ei[pos] = ent < N ? static_cast<int>(ent) : -1;
      }
      ncand += __popc(who);
    }
  }
  __syncwarp();
  // flag values (any non-zero value sends the row to the exact scan): 1 a list overflowed, 2 too many candidates,
  // 3 fewer than k candidates, 4 the proof failed
  const int why = overflow ? 1 : (ncand > kTkRescoreMax ? 2 : (ncand < k ? 3 : 0));
  if (why) { if (lane == 0) flag[row] = why; return; }
  // exact scores: the whole warp on one candidate -- its 512-byte row in ONE coalesced load -- sixteen candidates (8 KB of
  // row reads) in flight per warp
  constexpr int U = 16;
  for (int c0 = 0; c0 < ncand; c0 += U) {
    float d[U]; int id[U];
#pragma unroll
    for (int u = 0; u < U; ++u) id[u] = c0 + u < ncand ? ei[c0 + u] : -1;
    float4 tv[U];
#pragma unroll
    for (int u = 0; u < U; ++u)
      tv[u] = id[u] >= 0 ? __ldg(reinterpret_cast<const float4*>(table + static_cast<long long>(id[u]) * 128) + lane)
                         : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int u = 0; u < U; ++u) d[u] = qv.x * tv[u].x + qv.y * tv[u].y + qv.z * tv[u].z + qv.w * tv[u].w;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
      for (int u = 0; u < U; ++u) d[u] += __shfl_xor_sync(0xffffffffu, d[u], o);
    }
    float dv = d[0]; int iv = id[0];
#pragma unroll
    for (int u = 1; u < U; ++u) if (lane == u) { dv = d[u]; iv = id[u]; }
    if (lane < U && c0 + lane < ncand) es[c0 + lane] = iv >= 0 ? dv * inv_t[iv] : -3.0e38f;
  }
  __syncwarp();
  float kth = -3.0e38f;
  for (int r = 0; r < k; ++r) {
    float best = -3.0e38f; int bi = 0x7fffffff, bc = -1;
    for (int c = lane; c < ncand; c += 32) {
      const float s = es[c]; const int idx = ei[c];
      if (idx >= 0 && (s > best || (s == best && idx < bi))) { best = s; bi = idx; bc = c; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ob = __shfl_xor_sync(0xffffffffu, best, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o), oc = __shfl_xor_sync(0xffffffffu, bc, o);
      if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; bc = oc; }
    }
    if (lane == 0) {
      out_idx[row * k + r] = bc >= 0 ? bi : -1;
      out_score[row * k + r] = best;
      if (bc >= 0) ei[bc] = -1;   // taken
    }
    kth = best;
    __syncwarp();
  }
  // nothing outside the candidate set can reach the k-th exact score: its bf16 score is <= tau
  if (lane == 0) flag[row] = (kth > tau[row] + tk_err(err_q[row], err_t)) ? 0 : 4;   // (e_q: topk_tau_kernel)
}

// ------------------------------------------------------------------------------------------------ general path: select
// The k best of a row of exact scores [N] (general path: the fp32 GEMM's raw dot products, the row norms applied here),
// for any k <= 512, without a per-thread candidate list: a 4096-bin histogram of the scores (cosines: linear bins over
// [-1, 1]) gives the bin T that holds the k-th best; everything in the bins above it and in T itself -- k + a handful of
// entries -- is collected into shared memory and sorted (bitonic, score descending, ties: lower index first).  A crowded
// bin T (scores closer together than 5e-4) is split once more into 4096 sub-bins (1.2e-7 wide); a row that still does not
// fit the 2048-entry buffer -- thousands of identical scores -- is flagged and left to topk_exact_kernel.  Two or three
// coalesced reads of the row instead of O(k) shared-memory work per entity: k = 100 at B = 4096 took 31 ms in
// topk_exact_kernel (k = 512 at B = 256: 51 ms).
constexpr int kSelBins = 4096, kSelCap = 2048, kSelThreads = 256;
// The three passes over a row must put every score into the SAME bin each time: the arithmetic is spelled with the
// round-to-nearest intrinsics, which the compiler never contracts into an FMA (with `(r * iq * it + 1) * 2048` it fused the
// last product into the add in one loop and not in another: one entry counted and not collected).
__device__ __forceinline__ float tk_score(float raw, float iq, float it) { return __fmul_rn(__fmul_rn(raw, iq), it); }
__device__ __forceinline__ int tk_bin(float s, float& x) {
  x = __fmul_rn(__fadd_rn(s, 1.f), static_cast<float>(kSelBins / 2));
  return min(kSelBins - 1, max(0, static_cast<int>(x)));
}
__device__ __forceinline__ int tk_subbin(float x, int b) {
  return min(kSelBins - 1, max(0, static_cast<int>(__fmul_rn(__fsub_rn(x, static_cast<float>(b)), static_cast<float>(kSelBins)))));
}
// hist[] holds counts per bin; finds the largest bin t with count(bins >= t) >= need (need >= 1, total >= need):
// *out_t = t, *out_above = count(bins > t).  All threads call; results valid after the trailing barrier.
__device__ __forceinline__ void tk_find_bin(const unsigned* hist, int need, int* wsum, int* out_t, int* out_above) {
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  constexpr int kPer = kSelBins / kSelThreads;            // 16 bins per thread, thread 0 owns the TOP bins
  const int top = kSelBins - 1 - tid * kPer;
  int local = 0;
#pragma unroll
  for (int j = 0; j < kPer; ++j) local += static_cast<int>(hist[top - j]);
  int incl = local;                                        // inclusive scan over threads (top-down)
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
  if (lane == 31) wsum[w] = incl;
  __syncthreads();
  int base = 0;
  for (int j = 0; j < w; ++j) base += wsum[j];
  const int above = base + incl - local;                   // entries in bins above this thread's range
  if (above < need && above + local >= need) {
    int acc = above;
    for (int j = 0; j < kPer; ++j) {
      const int c = static_cast<int>(hist[top - j]);
      if (acc + c >= need) { *out_t = top - j; *out_above = acc; break; }
      acc += c;
    }
  }
  __syncthreads();
}

__global__ void __launch_bounds__(kSelThreads) topk_select_kernel(const float* __restrict__ raw, const float* __restrict__ inv_q,
                                                                  const float* __restrict__ inv_t, long long N, int k, long long n_rows,
                                                                  long long* __restrict__ out_idx, float* __restrict__ out_score,
                                                                  int* __restrict__ flag) {
  __shared__ unsigned hist[kSelBins];
  __shared__ float cs[kSelCap];
  __shared__ int ci[kSelCap];
  __shared__ int wsum[kSelThreads / 32];
  __shared__ int s_t, s_above, s_t2, s_above2, s_cnt;
  const int tid = threadIdx.x;
  for (long long row = blockIdx.x; row < n_rows; row += gridDim.x) {
    const float iq = inv_q[row];
    const float* r = raw + row * N;
    for (int b = tid; b < kSelBins; b += kSelThreads) hist[b] = 0u;
    if (tid == 0) { s_cnt = 0; s_t2 = -1; s_above2 = 0; }
    __syncthreads();
    for (long long e = tid; e < N; e += kSelThreads) {
      float x;
      atomicAdd(&hist[tk_bin(tk_score(r[e], iq, inv_t[e]), x)], 1u);
    }
    __syncthreads();
    tk_find_bin(hist, k, wsum, &s_t, &s_above);
    const int T = s_t, above = s_above;
    const bool crowded = above + static_cast<int>(hist[T]) > kSelCap;
    __syncthreads();
    if (crowded) {   // split bin T once more: the k - above best of ITS entries
      for (int b = tid; b < kSelBins; b += kSelThreads) hist[b] = 0u;
      __syncthreads();
      for (long long e = tid; e < N; e += kSelThreads) {
        float x;
        const int b = tk_bin(tk_score(r[e], iq, inv_t[e]), x);
        if (b == T) atomicAdd(&hist[tk_subbin(x, b)], 1u);
      }
      __syncthreads();
      tk_find_bin(hist, k - above, wsum, &s_t2, &s_above2);
    }
    const int T2 = s_t2;
    const int total = crowded ? above + s_above2 + static_cast<int>(hist[T2]) : above + static_cast<int>(hist[T]);
    if (total > kSelCap) {     // (uniform) thousands of equal scores at the cut: the exact kernel takes the row
      if (tid == 0) flag[row] = 1;
      __syncthreads();
      continue;
    }
    for (long long e = tid; e < N; e += kSelThreads) {
      float x;
      const float s = tk_score(r[e], iq, inv_t[e]);
      const int b = tk_bin(s, x);
      if (b > T || (b == T && (!crowded || tk_subbin(x, b) >= T2))) {
        const int pos = atomicAdd(&s_cnt, 1);
        cs[pos] = s; ci[pos] = static_cast<int>(e);
      }
    }
    __syncthreads();
    int P = 1;
    while (P < total) P <<= 1;
    for (int i = min(total, s_cnt) + tid; i < P; i += kSelThreads) { cs[i] = -3.0e38f; ci[i] = 0x7fffffff; }   // s_cnt == total
    __syncthreads();
    // bitonic sort: score descending, equal scores by ascending index
    for (int size = 2; size <= P; size <<= 1) {
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        for (int i = tid; i < (P >> 1); i += kSelThreads) {
          const int lo = ((i / stride) * (stride << 1)) + (i % stride), hi = lo + stride;
          const bool first_half = ((lo & size) == 0);      // this block of `size` sorts "best first"; the next one reversed
          const float a = cs[lo], bq = cs[hi];
          const int ai = ci[lo], bi = ci[hi];
          const bool a_before_b = a > bq || (a == bq && ai < bi);
          if (a_before_b != first_half) { cs[lo] = bq; cs[hi] = a; ci[lo] = bi; ci[hi] = ai; }
        }
        __syncthreads();
      }
    }
    for (int j = tid; j < k; j += kSelThreads) {
      out_idx[row * k + j] = j < total ? ci[j] : -1;
      out_score[row * k + j] = j < total ? cs[j] : -3.0e38f;
    }
    if (tid == 0) flag[row] = 0;
    __syncthreads();
  }
}

// Exact selection, one CTA per row: every thread keeps the k best of its entities, the CTA merges (k rounds of a block
// arg-max; ties: lower index first).  Two uses: rows whose flag is set after the filter path (always == 0; the scores
// are computed here, fp32 SIMT over N x E -- slow by design, the proof fails rarely), and the general path
// (always == 1, raw != nullptr: the row's raw dot products [N] come from the fp32 GEMM, the row norms are applied here).
__global__ void __launch_bounds__(256) topk_exact_kernel(const float* __restrict__ q, const float* __restrict__ inv_q,
                                                         const float* __restrict__ table, const float* __restrict__ inv_t, long long N,
                                                         int E, int k, const int* __restrict__ flag, int always,
                                                         const float* __restrict__ raw, long long* __restrict__ out_idx,
                                                         float* __restrict__ out_score, long long n_rows) {
  extern __shared__ uint8_t sm[];
  pdl_launch_dependents();
  pdl_wait();
  // a CTA takes rows blockIdx.x, blockIdx.x + gridDim.x, ...: after the filter path nearly every row is proven and the
  // launch is a few hundred CTAs that read their rows' flags and leave
  for (long long row = blockIdx.x; row < n_rows; row += gridDim.x) {
  if (!always && flag[row] == 0) continue;
  const int nt = blockDim.x;
  float* qn = reinterpret_cast<float*>(sm);                 // [E]
  float* ms = qn + E;                                       // [nt * k] kept candidates
  int* mi = reinterpret_cast<int*>(ms + nt * k);
  const float iq = inv_q[row];
  for (int c = threadIdx.x; c < E; c += nt) qn[c] = q[row * E + c] * iq;
  __syncthreads();
  // candidate j of thread t lives at [j * nt + t]: a warp's accesses to "its j-th candidates" hit 32 different banks
  // (thread-major [t * k + j] is an 8-way bank conflict at k = 100 and made a 4096-row call 35 ms)
  float* mys = ms + threadIdx.x; int* myi = mi + threadIdx.x;
  for (int j = 0; j < k; ++j) { mys[j * nt] = -3.0e38f; myi[j * nt] = -1; }
  float tau = -3.0e38f;
  int filled = 0;
  for (long long e = threadIdx.x; e < N; e += nt) {
    const float it = inv_t[e];
    float d = 0.f;
    if (raw != nullptr) {
      d = raw[row * N + e] * iq * it;
    } else {
      const float* tr = table + e * E;
      for (int c = 0; c < E; c += 4) {
        const float4 tv = *reinterpret_cast<const float4*>(tr + c);
        d += qn[c] * (tv.x * it) + qn[c + 1] * (tv.y * it) + qn[c + 2] * (tv.z * it) + qn[c + 3] * (tv.w * it);
      }
    }
    if (filled < k) {              // the first k entities of a thread are simply kept
      mys[filled * nt] = d; myi[filled * nt] = static_cast<int>(e); ++filled;
      if (filled == k) { float mn = mys[0]; for (int j = 1; j < k; ++j) mn = fminf(mn, mys[j * nt]); tau = mn; }
    } else if (d > tau) {          // replace this thread's smallest; the new smallest comes out of the same scan
      // among equal smallest scores the highest index goes (ties: lower index first); slots are not in index order
      int at = 0, ai = myi[0]; float mn = mys[0], mn2 = 3.0e38f;
      for (int j = 1; j < k; ++j) {
        const float v = mys[j * nt];
        const int vi = myi[j * nt];
        if (v < mn || (v == mn && vi > ai)) { mn2 = mn; mn = v; at = j; ai = vi; } else mn2 = fminf(mn2, v);
      }
      mys[at * nt] = d; myi[at * nt] = static_cast<int>(e);
      tau = fminf(mn2, d);
    }
  }
  __syncthreads();
  // k rounds of a block-wide arg-max over the kept candidates (thread 0 does the final step)
  __shared__ float rs[8]; __shared__ int ri[8], rc[8];
  const int nw = nt >> 5;
  for (int r = 0; r < k; ++r) {
    float best = -3.0e38f; int bi = 0x7fffffff, bc = -1;
    for (int c = threadIdx.x; c < nt * k; c += nt) {
      const float s = ms[c]; const int idx = mi[c];
      if (idx >= 0 && (s > best || (s == best && idx < bi))) { best = s; bi = idx; bc = c; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ob = __shfl_xor_sync(0xffffffffu, best, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o), oc = __shfl_xor_sync(0xffffffffu, bc, o);
      if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; bc = oc; }
    }
    if ((threadIdx.x & 31) == 0) { rs[threadIdx.x >> 5] = best; ri[threadIdx.x >> 5] = bi; rc[threadIdx.x >> 5] = bc; }
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int j = 1; j < nw; ++j)
        if (rs[j] > best || (rs[j] == best && ri[j] < bi)) { best = rs[j]; bi = ri[j]; bc = rc[j]; }
      out_idx[row * k + r] = bc >= 0 ? bi : -1;
      out_score[row * k + r] = best;
      if (bc >= 0) mi[bc] = -1;
    }
    __syncthreads();
  }
  }   // rows of this CTA
}

}  // namespace pbg
