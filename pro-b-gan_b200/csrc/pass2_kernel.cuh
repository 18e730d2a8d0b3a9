// pass2_kernel.cuh -- the generator + discriminator pass as ONE persistent kernel of CTA PAIRS (cta_group::2).
//
//   gather/concat -> G.L0 -> G.L1 -> G.L2 (tanh, cosine)         (pro_b_gan_infer.py:186-188, :201-202)
//                 -> D.L0 -> D.L1 (+ final H/2 -> 1 dot, sigmoid) (pro_b_gan_infer.py:207, :302)
//
// Activations are handed from layer to layer through L2 (bf16, row-major) with per-row-block arrival counters in
// global memory: no grid-wide barrier, no launch per layer.  The tiling is cut for the L2 -> SM operand bandwidth:
// two CTAs on one TPC form a pair and compute one 256-row x BLOCK_N tile with tcgen05.mma.cta_group::2
// (M = 256: 128 rows of A per CTA; the BLOCK_N rows of W are split in halves, one per CTA), so a 64-deep k-block
// costs each SM 16 KB of A + 16 KB of W (64 B/clk at full MMA rate) instead of 48 KB (96 B/clk) for a single-CTA
// 128 x 256 tile, against ~70 B/clk/SM that the L2 fabric delivers chip-wide (profiles/ubench_r1_*.txt).  This main
// loop alone sustains 513-546 clk per k-block on all 148 SMs (floor 512; tools/ubench_pipe.cu); inside this kernel the
// K = 1024 tiles run at 555-590 in a lone 48-SM pass and 595-660 with 148 SMs busy (-DPBG_KB_PROBE=1; DESIGN.md 3.1).
//
//   leader CTA (cluster rank 0)                               peer CTA (rank 1)
//   warps 0..7  epilogue of its 128 rows / gather groups      warps 0..7  epilogue of its 128 rows / gather groups
//   warp 8   TMA producer for its halves of A and W           warp 8   TMA producer for its halves of A and W,
//                                                                      signalling the leader's full barriers
//   warp 9   MMA issuer (one thread) for the pair             warp 9   scheduler (one thread): pops tickets up to a
//                                                                      ring's depth ahead, waits for the item's input
//                                                                      row block, publishes the item to both CTAs
//   (PBG_ROLES_FIRST=1 puts the two single-thread roles in warps 0 / 1, the round-1 layout; measured neutral)
//
// Tickets index a static, topologically ordered item list described by a few segments in the kernel parameters
// (layer by layer, row-block major).  A pair takes its tickets in order from one atomic counter and works through
// them in order, which makes any topological order deadlock-free (the unfinished item with the smallest ticket never
// waits on anything unfinished).  The scheduler polls an item's dependency counter before publishing it, so the
// producers never wait between an item's loads: every stage is refilled with W and A the moment it frees.
// The gather of every row is "phase 0" of the epilogue warps.
//
// A workspace row block that its consumer layer has finished with is dropped from L2 (discard.global.L2) by the epilogue
// warps that can prove it dead from the dependency counters, so dead activations are never written back to HBM (p2_discard).
//
// Epilogues: bias + LeakyReLU -> bf16 -> swizzled staging (double-buffered per warp) -> TMA store; the final
// discriminator dot and the cosine against the tail embedding are written as per-64-column partials that the last
// warp to arrive for the 256-row block sums in a fixed order (bit-identical for any batch size / interleaving).
#pragma once
#include <cuda.h>
#include "ptx.cuh"
#include "gather.cuh"
#include "tc_common.cuh"
#include "pass_common.cuh"

namespace pbg {

#ifndef PBG_STAGES
#define PBG_STAGES 5
#endif
#ifndef PBG_EPI_WARPS
#define PBG_EPI_WARPS 8
#endif
constexpr int kP2Stages = PBG_STAGES;      // operand ring depth (32 KB per stage and CTA)
constexpr int kP2Epi = PBG_EPI_WARPS;      // epilogue warps per CTA: 8 (two per TMEM lane quarter) or 16 (four; needs PBG_STAGES=4)
constexpr int kP2Slots = kP2Epi / 4;       // warps per lane quarter = 64-column chunks of a tile in flight per quarter
constexpr int kP2Threads = 64 + 32 * kP2Epi;
static_assert(kP2Epi == 8 || kP2Epi == 16, "epilogue warps");
// Warp roles.  The warp scheduler prefers the higher warp id among eligible warps (B300_MICROARCH.md: "hi-wid-first"),
// so the two single-thread roles everything else waits for -- the TMA producer and the MMA issuer / scheduler -- are
// the LAST two warps and the eight epilogue warps come first (PBG_ROLES_FIRST=1: the r1 layout, roles in warps 0 / 1).
#ifndef PBG_ROLES_FIRST
#define PBG_ROLES_FIRST 0
#endif
constexpr int kProdWarp = PBG_ROLES_FIRST ? 0 : kP2Epi;
constexpr int kMmaWarp = PBG_ROLES_FIRST ? 1 : kP2Epi + 1;
constexpr int kEpiWarp0 = PBG_ROLES_FIRST ? 2 : 0;            // first epilogue warp
constexpr int kTraceThread = kEpiWarp0 * 32;                  // the epilogue thread that writes the diagnostics
#ifndef PBG_P2RING
#define PBG_P2RING 4
#endif
constexpr int kP2Ring = PBG_P2RING;   // items the scheduler may run ahead of the workers (pre-claimed tickets per pair)
constexpr int kP2Rows = 256;                        // rows of one pair tile = one dependency block
constexpr int kP2GroupsPerBlock = kP2Rows / 4;      // 4-row gather groups per block
constexpr int kP2GatherPerBlock = 4;                // gather items per block: 64 rows = 16 warps x 4 rows
constexpr int kP2WarpsPerPair = 2 * kP2Epi;
constexpr int kMaxMirrors = 7;                      // peers of an 8-GPU box

// -DPBG_KB_PROBE=1 (diagnostics build, tools only): the MMA issuer of every leader CTA times its k-block loops per layer
// with two clock reads per TILE -- the production instance otherwise unchanged -- and launch 30 of a process prints them.
#ifndef PBG_KB_PROBE
#define PBG_KB_PROBE 0
#endif
#if PBG_KB_PROBE
__device__ int g_probe_n;
#endif

struct P2Layer {
  int num_kb;        // K / 64
  int block_n;       // UMMA N of this layer's pair tiles (128 / 256)
  int n_tiles;       // padded output width / block_n
  int epi;           // PEPI_*
  int dep_kind;      // DEP_* counter that gates this layer's A operand
  int out_kind;      // DEP_* counter this layer's stores bump, or -1
  int ldo;           // PEPI_STORE: leading dimension of out (elements)
  int bias_off;      // offset (floats) of this layer's bias in the shared-memory copy, or -1: read it from global
  const float* bias; // [n_tiles * block_n] fp32, zero padded
  __nv_bfloat16* out;// PEPI_STORE: next layer's A operand
};

// Static tickets from `start` up to the next segment.  Per row block rb = rb0 + i / (n_tiles + n_tiles2) the segment
// holds the n_tiles tiles of layer `kind` followed by the n_tiles2 tiles of layer `kind2` (n_tiles2 = 0: one layer).
struct P2Segment { int kind, n_tiles, start, rb0, kind2, n_tiles2; };

struct alignas(64) Pass2Params {
  CUtensorMap tm_a[5];  // A operand of layer i: xg0, xd0, actG0, actD0, actG1   (box 64 x 128 rows, SWIZZLE_128B)
  CUtensorMap tm_w[5];  // weights of layer i                                      (box 64 x block_n / 2 rows)
  CUtensorMap tm_o[5];  // PEPI_STORE layers: the activation buffer they write      (box 64 x 32 rows)
  P2Layer layer[5];
  GatherParams gather;
  unsigned layer_mask;
  int gather_defer;      // 1: a gather group's completion wait + arrival ride behind the next group's loads
  int gather_external;   // 1: xg0 / xd0 were written by a gather kernel before this launch (phase0_groups = 0)
  int gather_ahead;      // 1: the gather groups belong to the NEXT request (another staging slot): nothing in this pass waits
                         //    for them, no arrivals; the warps gather only when idle and drain the rest before they exit
  int no_deps;           // 1: single-layer launch (pbg_linear_bf16): the A operand is the caller's, nothing to wait for
  int discard;           // 1: dead workspace row blocks (activations and gathered rows the next layer has consumed) are
                         //    dropped from L2 with discard.global.L2 instead of being written back to HBM when evicted
  const void* dead_xg;   // discard: the first-layer operand buffers of THIS pass when nothing will read them again (the
  const void* dead_xd;   //    ctx's own gather buffers, or the staging slot a stage-next pass consumes), else null
  int dead_ldg, dead_ldd;
  int poll_ns;
  int phase0_groups;    // 4-row gather groups (every row of the pass), done by the epilogue warps before their first tile
  int n_total;          // tickets of this launch
  int n_seg;
  P2Segment seg[16];
  int nrb;              // 256-row blocks in this pass
  int rb_cap;           // stride of the counter arrays
  int M;                // rows in this pass
  float slope;
  PassSched* sched;
  int* ready;           // [DEP_KINDS][rb_cap]
  int* fin;             // [FIN_KINDS][rb_cap]
  // generator output (PEPI_TANH)
  void* gen_out; int out_f32; int n_valid; int ld_gen;
  float* cosine; const float* tail_tab; const long long* tail_idx; long long tail_stride; long long n_ent;
  float* part_g;        // [nrb][slots_g][3][256]
  int slots_g;
  // discriminator output (PEPI_ROWDOT)
  const float* w3; float b3; float* logits; float* probs;
  int w3_off;           // offset (floats) of w3 in the shared-memory copy, or -1
  float* part_d;        // [nrb][slots_d][256]
  int slots_d;
  // result mirrors: the same rows of every result are also written to these buffers (peer GPUs' windows over NVLink:
  // the output all-gather of a batch-sharded job without a collective; pbg_set_result_mirrors)
  int n_mirror;
  void* mir_gen[kMaxMirrors]; float* mir_cos[kMaxMirrors]; float* mir_logits[kMaxMirrors]; float* mir_probs[kMaxMirrors];
  // result multicast: NVSwitch multicast addresses of the same result buffers (pbg_set_result_multicast): one
  // multimem.st per 16 bytes leaves this GPU and the switch replicates it into every GPU's copy
  void* mc_gen; float* mc_cos; float* mc_logits; float* mc_probs;
  long long* trace;
};
static_assert(sizeof(Pass2Params) <= 4096, "kernel parameter space");

struct P2Smem {
  static constexpr int kA = 128 * kBlockK * 2;
  static constexpr int kW = 128 * kBlockK * 2;   // this CTA's half of a 256-wide W tile
  static constexpr int kStage = kA + kW;
  static constexpr int kStagingOff = kP2Stages * kStage;
  static constexpr int kStagingPerWarp = 4096;   // one 32 x 64 bf16 store tile / one 32 x 32 fp32 transpose tile
  static constexpr int kBiasOff = kStagingOff + kP2Epi * kStagingPerWarp;
  static constexpr int kBiasFloats = 6144;       // every layer's padded bias + the final dot weights, when they fit
  static constexpr int kBarOff = kBiasOff + kBiasFloats * 4;
  static constexpr int kXchgOff = kBarOff + 256;          // cosine partials handed between the two warps of a quarter
  static constexpr int kXchgBytes = 4 * 32 * 3 * 4;
  static constexpr int kTotal = kXchgOff + kXchgBytes + 256 + 1024 /*alignment slack*/;
};
static_assert(P2Smem::kTotal <= 232448, "pass2: shared memory budget");

__device__ __forceinline__ void st_cluster_u32x2(uint32_t cluster_addr, uint2 v) {
  asm volatile("st.shared::cluster.v2.u32 [%0], {%1, %2};" ::"r"(cluster_addr), "r"(v.x), "r"(v.y) : "memory");
}
// Stores to an NVSwitch multicast address: every replica (one per GPU of the multicast group) receives the value.
__device__ __forceinline__ void multimem_st_v4(void* mc_addr, uint4 v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc_addr), "f"(__uint_as_float(v.x)),
               "f"(__uint_as_float(v.y)), "f"(__uint_as_float(v.z)), "f"(__uint_as_float(v.w)) : "memory");
}
__device__ __forceinline__ void multimem_st_f32(float* mc_addr, float v) {
  asm volatile("multimem.st.relaxed.sys.global.f32 [%0], %1;" ::"l"(mc_addr), "f"(v) : "memory");
}
__device__ __forceinline__ float2 add2(float2 a, float2 b) {
  float2 d;
  asm("{\n\t.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tadd.rn.f32x2 rd, ra, rb;\n\t"
      "mov.b64 {%0, %1}, rd;\n\t}\n"
      : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
  return d;
}
__device__ __forceinline__ float2 mul2(float2 a, float2 b) {
  float2 d;
  asm("{\n\t.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmul.rn.f32x2 rd, ra, rb;\n\t"
      "mov.b64 {%0, %1}, rd;\n\t}\n"
      : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
  return d;
}
// bf16x2( leaky(a + b) ): packed fp32 add and multiply, scalar max, one packed convert
__device__ __forceinline__ uint32_t bias_leaky_pack(uint32_t a0, uint32_t a1, float b0, float b1, float slope) {
  const float2 y = add2(make_float2(__uint_as_float(a0), __uint_as_float(a1)), make_float2(b0, b1));
  const float2 s = mul2(y, make_float2(slope, slope));
  return pack_bf16x2(fmaxf(y.x, s.x), fmaxf(y.y, s.y));
}

__device__ __forceinline__ int p2_dep_target(const Pass2Params& p, int dep_kind) {
  if (p.no_deps) return 0;
  if (dep_kind == DEP_X) return p.gather_external ? 0 : kP2GroupsPerBlock;
  const int producer = dep_kind == DEP_G0 ? IT_G_L0 : (dep_kind == DEP_D0 ? IT_D_L0 : IT_G_L1);
  return p.layer[producer].n_tiles * kP2WarpsPerPair;
}
// A warp announces "my part of block rb of buffer dep_kind is in global memory".
//   generic stores (gather): the warp barrier orders every lane's stores before lane 0's release increment.
//   bulk stores (activations): lane 0 issued them; cp.async.bulk.wait_group 0 returns once they have been performed
//   (in L2, the point of coherence for every consumer, which reads them with TMA after a relaxed poll of the counter
//   and a proxy fence), so the increment itself is relaxed -- a release here is a MEMBAR.ALL.GPU on the critical path
//   of every layer-to-layer hand-off.
__device__ __forceinline__ void p2_arrive(const Pass2Params& p, int dep_kind, int rb, int lane, bool async_stores,
                                          long long* t_wait = nullptr) {
  __syncwarp();
  if (lane == 0) {
    int* ctr = p.ready + dep_kind * p.rb_cap + rb;
    if (async_stores) {
      const long long t0 = t_wait ? clock64() : 0;
      tma_store_wait<0>();
      if (t_wait) *t_wait += clock64() - t0;
      red_relaxed_gpu_add(ctr, 1);
    } else {
      red_release_gpu_add(ctr, 1);
    }
  }
}
// Arrival for data whose bulk stores have already completed (relaxed increment, see p2_arrive).
__device__ __forceinline__ void p2_arrive_done(const Pass2Params& p, int dep_kind, int rb, int lane) {
  if (lane == 0) red_relaxed_gpu_add(p.ready + dep_kind * p.rb_cap + rb, 1);
}
// A producer thread waits until block rb of buffer dep_kind is complete.  The data is read by
// TMA only (async proxy, from L2): the proxy fence orders the counter read before the bulk loads that follow.
__device__ __forceinline__ void p2_poll_dep(const Pass2Params& p, int dep_kind, int rb) {
  const int target = p2_dep_target(p, dep_kind);
  const int* ctr = p.ready + dep_kind * p.rb_cap + rb;
  uint32_t spins = 0;
  while (ld_relaxed_gpu(ctr) < target) {
    __nanosleep(p.poll_ns);
#if PBG_HANG_GUARD
    if (++spins > 4000000u) pbg_wait_timed_out("dependency (kind, row block)", dep_kind, rb);
#endif
  }
  fence_proxy_async_all();
}

// Workspace lines that nothing will read again (a row block of activations whose consumer layer has finished with it)
// are dirty in L2, and with several lanes' workspaces cycling through the cache they would be written back to HBM on
// eviction: tens of megabytes per pass that no one ever reads.  discard.global.L2 drops a 128-byte line without the
// write-back (SASS: CCTL.E.RML2).  Warp `part` of `nparts` takes every nparts-th 4 KB piece of [base, base + bytes).
__device__ __forceinline__ void p2_discard(const void* base, size_t bytes, int part, int nparts, int lane) {
  const char* b = static_cast<const char*>(base);
  for (size_t off = static_cast<size_t>(part) * 4096 + static_cast<size_t>(lane) * 128; off < bytes; off += static_cast<size_t>(nparts) * 4096)
    asm volatile("discard.global.L2 [%0], 128;" ::"l"(b + off) : "memory");
}

// Tail-embedding values of 32 columns for this warp's 32 rows: coalesced 16-byte loads (four rows per instruction),
// then into the warp's 4 KB staging tile (row r at r * 128 B, piece t at t ^ (r & 7)) for row-per-lane reads.
__device__ __forceinline__ void p2_tail_load(float4 (&tv)[8], unsigned long long trow_bits, int col0, int n_valid, int lane) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int r = i * 4 + (lane >> 3), t = lane & 7;
    const float* tp2 = reinterpret_cast<const float*>(__shfl_sync(0xffffffffu, trow_bits, r));
    tv[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (tp2 != nullptr && col0 + t * 4 < n_valid) tv[i] = ld_stream4(tp2 + col0 + t * 4);
  }
}
__device__ __forceinline__ void p2_tail_stage(uint8_t* st, const float4 (&tv)[8], int lane) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int r = i * 4 + (lane >> 3), t = lane & 7;
    *reinterpret_cast<float4*>(st + r * 128 + ((t ^ (r & 7)) << 4)) = tv[i];
  }
  __syncwarp();
}
// this lane's row against 32 generator outputs f[0..31] (columns col0 .. col0 + 31)
__device__ __forceinline__ void p2_tail_dot(const uint8_t* st, const float* f, int col0, int n_valid, int lane, float& d, float& pp,
                                            float& tt) {
#pragma unroll
  for (int t = 0; t < 8; ++t) {
    const float4 x = *reinterpret_cast<const float4*>(st + lane * 128 + ((t ^ (lane & 7)) << 4));
    if (col0 + t * 4 < n_valid) {
      d += f[4 * t] * x.x + f[4 * t + 1] * x.y + f[4 * t + 2] * x.z + f[4 * t + 3] * x.w;
      pp += f[4 * t] * f[4 * t] + f[4 * t + 1] * f[4 * t + 1] + f[4 * t + 2] * f[4 * t + 2] + f[4 * t + 3] * f[4 * t + 3];
      tt += x.x * x.x + x.y * x.y + x.z * x.z + x.w * x.w;
    }
  }
  __syncwarp();
}

// Gather group for the common layout (E = 128, Z <= 128, unpadded xg / xd rows): four rows through the warp's staging
// tile and out with bulk stores, so that the arrival can follow cp.async.bulk.wait_group (a few hundred clocks)
// instead of a release fence over 28 generic stores per lane.  Returns with lane 0's last bulk store committed but
// not waited for: the caller completes it (wait_group 0, then the arrival) -- `before_staging()` is called once this
// group's row loads are in flight and before the staging tile is written, which is where the caller completes the
// PREVIOUS group, so that a store's completion latency hides behind the next group's load latency.
// keep: the rows are for a LATER launch (the next request of a stage-next pass): they are stored with the evict-last L2
// policy, so that the traffic of the passes in between does not push them out to HBM and back.
template <class F>
__device__ __forceinline__ void p2_gather_group_bulk(const GatherParams& g, long long group, int lane, uint8_t* st,
                                                     F&& before_staging, bool keep) {
  const long long r0 = group * 4;
  __nv_bfloat16* xg = static_cast<__nv_bfloat16*>(g.xg);
  __nv_bfloat16* xd = static_cast<__nv_bfloat16*>(g.xd);
  const float* src = nullptr;
  bool bad = false;
  if (lane < 12) {   // lane l resolves the source row of (row l / 3, operand l % 3): 0 head, 1 relation, 2 tail
    const long long row = r0 + lane / 3;
    const int which = lane % 3;
    if (row < g.B) {
      if (which == 0) {
        if (g.heads) { long long i = g.heads[row * g.head_stride]; if (i < 0) i += g.N; if (i < 0 || i >= g.N) { bad = true; i = 0; } src = g.node_emb + i * g.E; }
        else src = g.h + row * g.E;
      } else if (which == 1) {
        if (g.rels) { long long i = g.rels[row * g.rel_stride]; if (i < 0 || i >= g.R) { bad = true; i = 0; } src = g.rel_emb + i * g.E; }
        else src = g.r + row * g.E;
      } else if (g.tails) {   // range-checked whenever tail ids are given: a generator-only pass reads them too (cosine)
        long long i = g.tails[row * g.tail_stride]; if (i < 0) i += g.N; if (i < 0 || i >= g.N) { bad = true; i = 0; } src = g.node_emb + i * g.E;
      } else if (xd != nullptr) {
        src = g.t + row * g.E;
      }
    }
  }
  if (bad) atomicOr(g.err_flag, 1);
  const unsigned long long sp = reinterpret_cast<unsigned long long>(src);
  const int Z4 = g.Z >> 2;
  const int wg = 2 * g.E + g.Z, wd = 3 * g.E;            // row widths (elements) = ldg / ldd on this path
  float4 hv[4], rv[4], tv[4], zv[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float* ph = reinterpret_cast<const float*>(__shfl_sync(0xffffffffu, sp, j * 3 + 0));
    const float* pr = reinterpret_cast<const float*>(__shfl_sync(0xffffffffu, sp, j * 3 + 1));
    const float* pt = reinterpret_cast<const float*>(__shfl_sync(0xffffffffu, sp, j * 3 + 2));
    const long long row = r0 + j;
    hv[j] = rv[j] = tv[j] = zv[j] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row < g.B) {
      hv[j] = ld_stream4(ph + 4 * lane);
      rv[j] = ld_stream4(pr + 4 * lane);
      if (xd != nullptr) tv[j] = ld_stream4(pt + 4 * lane);
      if (xg != nullptr && lane < Z4) zv[j] = ld_stream4(g.z + row * g.Z + 4 * lane);
    }
  }
  before_staging();
  const long long nrow = min(4ll, g.B - r0);   // rows of a group are consecutive in xg / xd: one bulk store each
  // the staging tile holds one of the two outputs at a time (4 x 640 B, then 4 x 768 B)
  if (xg != nullptr) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(st) + j * wg;
      store4<__nv_bfloat16>(o + 4 * lane, hv[j]);
      store4<__nv_bfloat16>(o + g.E + 4 * lane, rv[j]);
      if (lane < Z4) store4<__nv_bfloat16>(o + 2 * g.E + 4 * lane, zv[j]);
    }
    fence_proxy_async_smem();
    __syncwarp();
    if (lane == 0 && nrow > 0) {
      if (keep) bulk_store_1d_hint(xg + r0 * wg, st, static_cast<uint32_t>(nrow * wg * 2), kEvictLast);
      else bulk_store_1d(xg + r0 * wg, st, static_cast<uint32_t>(nrow * wg * 2));
      tma_store_commit();
      if (xd != nullptr) tma_store_wait_read<0>();
    }
    __syncwarp();
  }
  if (xd != nullptr) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(st) + j * wd;
      store4<__nv_bfloat16>(o + 4 * lane, hv[j]);
      store4<__nv_bfloat16>(o + g.E + 4 * lane, rv[j]);
      store4<__nv_bfloat16>(o + 2 * g.E + 4 * lane, tv[j]);
    }
    fence_proxy_async_smem();
    __syncwarp();
    if (lane == 0 && nrow > 0) {
      if (keep) bulk_store_1d_hint(xd + r0 * wd, st, static_cast<uint32_t>(nrow * wd * 2), kEvictLast);
      else bulk_store_1d(xd + r0 * wd, st, static_cast<uint32_t>(nrow * wd * 2));
      tma_store_commit();
    }
  }
}

// ------------------------------------------------------------------------------------------------ the kernel
// Always 0 (an item's bits 24..31 are never set), but only known at run time: added to the address of a consumer's
// sched_empty arrive so that the arrive cannot be issued before the load of the ring slot has returned.
__device__ __forceinline__ uint32_t ring_dep(uint2 it) { return (it.x >> 24) << 3; }

// TR: the diagnostics instance (pbg_debug_trace); the production instance carries no trace code or registers.
// FASTG: the gather only carries the E = 128, Z <= 128 register path (the host checks the dims).
// BIASS: biases + final dot weights are copied to shared memory in the prologue (they fit for H <= 1024); without it
//        (wide models: long main loops, the epilogue is off the critical path) they are read through the global path.
template <bool TR, bool FASTG, bool BIASS>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kP2Threads, 1)
pbg_pass2_kernel(const __grid_constant__ Pass2Params p) {
  using L = P2Smem;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::kBarOff);
  uint64_t* empty_bar = full_bar + kP2Stages;
  uint64_t* tmem_full = empty_bar + kP2Stages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint64_t* sched_full = tmem_empty + 2;
  uint64_t* sched_empty = sched_full + kP2Ring;
  uint64_t* bias_bar = sched_empty + kP2Ring;
  uint2* ring = reinterpret_cast<uint2*>(bias_bar + 1);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(ring + kP2Ring);
  int* last_flag = reinterpret_cast<int*>(tmem_slot + 1);
  volatile long long* t_issue = reinterpret_cast<volatile long long*>(smem + L::kXchgOff + L::kXchgBytes);  // [kP2Stages], diagnostics
  float* xchg = reinterpret_cast<float*>(smem + L::kXchgOff);
  float* sbias = reinterpret_cast<float*>(smem + L::kBiasOff);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const long long t_entry = (TR && p.trace && threadIdx.x == 0) ? static_cast<long long>(globaltimer_ns()) : 0;
  // Programmatic dependent launch: the next pass may start its prologue while this one is still running ...
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  constexpr int kRingConsumers = 2 * (1 + kP2Epi) + 1;  // both producers, the MMA issuer, 16 epilogue warps

  if (threadIdx.x == 0) {
    for (int i = 0; i < 5; ++i) {
      if (p.layer_mask & (1u << i)) {
        prefetch_tmap(&p.tm_a[i]);
        prefetch_tmap(&p.tm_w[i]);
        if (p.layer[i].epi == PEPI_STORE) prefetch_tmap(&p.tm_o[i]);
      }
    }
    for (int s = 0; s < kP2Stages; ++s) {
      mbar_init(&full_bar[s], 1);     // leader's: its producer's arrive.expect_tx (bytes of both CTAs)
      mbar_init(&empty_bar[s], 1);    // tcgen05.commit, multicast to both CTAs
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tmem_full[s], 1);                  // tcgen05.commit, multicast
      mbar_init(&tmem_empty[s], kP2WarpsPerPair);   // leader's: the epilogue warps of both CTAs
    }
    for (int s = 0; s < kP2Ring; ++s) {
      mbar_init(&sched_full[s], 1);                 // the scheduler (local + remote arrive)
      mbar_init(&sched_empty[s], kRingConsumers);   // peer's (the scheduler's CTA)
    }
    mbar_init(bias_bar, 1);
    fence_mbar_init();
    if (BIASS) {
    // Biases (and the final dot weights) live in shared memory for the whole launch: with ~224 KB of the SM carved out
    // as shared memory a bias read through the global path is an L2 round trip.  One bulk copy per array, in flight
    // while the rest of the prologue and the gather run; the epilogue warps wait for them once.
    uint32_t bytes = 0;
    for (int k = 0; k < 5; ++k)
      if (p.layer_mask & (1u << k)) bytes += static_cast<uint32_t>(p.layer[k].n_tiles * p.layer[k].block_n) * 4u;
    if (p.layer_mask & (1u << IT_D_L1)) bytes += static_cast<uint32_t>(p.layer[IT_D_L1].n_tiles * p.layer[IT_D_L1].block_n) * 4u;
    mbar_arrive_expect_tx(bias_bar, bytes);
    for (int k = 0; k < 5; ++k)
      if (p.layer_mask & (1u << k))
        bulk_load_1d(sbias + p.layer[k].bias_off, p.layer[k].bias, static_cast<uint32_t>(p.layer[k].n_tiles * p.layer[k].block_n) * 4u, bias_bar);
    if (p.layer_mask & (1u << IT_D_L1))
      bulk_load_1d(sbias + p.w3_off, p.w3, static_cast<uint32_t>(p.layer[IT_D_L1].n_tiles * p.layer[IT_D_L1].block_n) * 4u, bias_bar);
    }
  }
  if (warp == kMmaWarp) tmem_alloc_pair<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  // ... and this pass waits here, prologue done, until the previous grid (which shares the workspace, the counters
  // and the scheduler) has completed.  Everything above touches only this CTA and the immutable weights.
  asm volatile("griddepcontrol.wait;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;
  long long* const clk0 = reinterpret_cast<long long*>(smem + L::kXchgOff + L::kXchgBytes) + 8;   // [2], behind the diagnostics' t_issue[]
  if (blockIdx.x == 0 && threadIdx.x == 0) { clk0[0] = clock64(); clk0[1] = static_cast<long long>(globaltimer_ns()); }
  long long* const tr = (TR && p.trace) ? p.trace + kTraceSlots * blockIdx.x : nullptr;
  if (tr && threadIdx.x == 0) { tr[0] = clock64(); tr[14] = static_cast<long long>(globaltimer_ns()); tr[254] = t_entry; }

  const uint32_t lead_tmem_empty = mapa_u32(smem_u32(tmem_empty), 0);    // the leader's, as seen from either CTA
  const uint32_t sched_empty_addr = mapa_u32(smem_u32(sched_empty), 1);  // the scheduler CTA's
  const uint32_t ring_addr = mapa_u32(smem_u32(ring), 1);
  if (warp == kMmaWarp && !leader) {
    // ------------------------------------------------------------ scheduler (one thread of the peer CTA)
    if (lane == 0) {
      uint32_t slot = 0, sphase = 0;
      const uint32_t lead_sched_full = mapa_u32(smem_u32(sched_full), 0);
      for (;;) {
        const int ticket = atomicAdd(&p.sched->q_head, 1);
        uint2 it = make_uint2(IT_END, 0u);
        if (ticket < p.n_total) {
          int sg = 0;
          while (sg + 1 < p.n_seg && ticket >= p.seg[sg + 1].start) ++sg;
          const int i = ticket - p.seg[sg].start;
          const int nt1 = p.seg[sg].n_tiles, nt = nt1 + p.seg[sg].n_tiles2;
          const int j = i % nt;
          it = make_uint2(static_cast<uint32_t>(j < nt1 ? p.seg[sg].kind : p.seg[sg].kind2) | (static_cast<uint32_t>(j < nt1 ? j : j - nt1) << 8),
                          static_cast<uint32_t>(p.seg[sg].rb0 + i / nt));
        }
        // Ring protocol: the item lives in this (the scheduler's) CTA only; the leader's consumers fetch it with a
        // remote load after their own sched_full barrier fires.  All arrives use CTA-scope release (a cluster-scope
        // release is a MEMBAR.ALL.GPU in front of every arrive): the slot is written to local shared memory before
        // the remote arrive leaves this SM, and a consumer's arrive on sched_empty carries a data dependency on its
        // load of the slot.
        // The scheduler, not the producer, waits for the item's A operand (the row block of the previous layer, or the
        // gathered rows): it runs up to a ring ahead of the workers, so the wait costs nothing in steady state, every
        // item in the ring is ready, and the producers refill each stage with W and A the moment it frees.  (A
        // producer that polls between an item's loads delays the A loads of the first ring's worth of K-blocks until
        // the previous item's LAST stage has freed, and its proxy fence then waits for its own bulk loads in flight:
        // 3-4 thousand clocks of tensor-pipe idle per tile boundary, tools/ubench_pipe.cu vs the r1f trace.)
        if ((it.x & 0xff) != IT_END) p2_poll_dep(p, p.layer[it.x & 0xff].dep_kind, static_cast<int>(it.y));
        mbar_wait_role(&sched_empty[slot], sphase ^ 1);
        ring[slot] = it;
        mbar_arrive(&sched_full[slot]);
        mbar_arrive_cluster(lead_sched_full + slot * 8);  // release at cluster scope: the slot is visible to the remote loads
        if (++slot == kP2Ring) { slot = 0; sphase ^= 1; }
        if ((it.x & 0xff) == IT_END) break;
      }
    }
    __syncwarp();
  } else if (warp == kProdWarp) {
    // ------------------------------------------------------------ TMA producer (both CTAs)
    if (lane == 0) {
      uint32_t stage = 0, phase = 0, slot = 0, sphase = 0;
      long long w_dep = 0, w_empty = 0, n_items = 0;
      const uint32_t lead_full = mapa_u32(smem_u32(full_bar), 0);
      for (;;) {
        mbar_wait_role(&sched_full[slot], sphase);
        const uint2 it = ld_cluster_u32x2(ring_addr + slot * 8);
        mbar_arrive_remote(sched_empty_addr + slot * 8 + ring_dep(it));
        if (++slot == kP2Ring) { slot = 0; sphase ^= 1; }
        const int kind = it.x & 0xff;
        if (kind == IT_END) break;
        long long* ti = (tr && n_items < kTraceItems) ? tr + 16 + 4 * n_items : nullptr;
        if (ti) { ti[0] = (clock64() << 20) | (static_cast<long long>(it.y & 0xfff) << 8) | kind; }
        ++n_items;
        const int n_blk = (it.x >> 8) & 0xff;
        const int rb = static_cast<int>(it.y);
        const P2Layer& ly = p.layer[kind];
        const int w_rows = ly.block_n >> 1;
        const uint32_t bytes_pair = 2u * (L::kA + static_cast<uint32_t>(w_rows) * kBlockK * 2);
        const int a_row = rb * kP2Rows + static_cast<int>(rank) * 128;
        const int w_row = n_blk * ly.block_n + static_cast<int>(rank) * w_rows;
        for (int kb = 0; kb < ly.num_kb; ++kb) {
          if (tr) { const long long t = clock64(); mbar_wait_role(&empty_bar[stage], phase ^ 1); w_empty += clock64() - t; }
          else mbar_wait_role(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem + stage * L::kStage;
          if (leader) mbar_arrive_expect_tx(&full_bar[stage], bytes_pair);
          if (tr) t_issue[stage] = clock64();
          tma_load_2d_pair(sa + L::kA, &p.tm_w[kind], lead_full + stage * 8, kb * kBlockK, w_row);
          tma_load_2d_pair(sa, &p.tm_a[kind], lead_full + stage * 8, kb * kBlockK, a_row);
          if (++stage == kP2Stages) { stage = 0; phase ^= 1; }
        }
      }
      if (tr) { tr[1] = w_empty; tr[2] = clock64(); tr[12] = n_items; if (leader) tr[11] = w_dep; }
    }
    __syncwarp();
  } else if (warp == kMmaWarp) {
    // ------------------------------------------------------------ MMA issuer (one thread of the leader CTA)
    if (lane == 0) {
      uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0, slot = 0, sphase = 0;
      long long w_full = 0, w_tmem = 0, w_item = 0, n_kb = 0, lat_sum = 0, lat_n = 0, lat_max = 0;
      int n_it = 0;
#if PBG_KB_PROBE
      long long pr_clk[5] = {0, 0, 0, 0, 0}, pr_item = 0, pr_tmem = 0;
      int pr_tiles[5] = {0, 0, 0, 0, 0};
      const long long pr_begin = clock64();
#endif
      for (;;) {
#if PBG_KB_PROBE
        const long long pr_t0 = clock64();
#endif
        if (tr) { const long long t = clock64(); mbar_wait_role(&sched_full[slot], sphase); w_item += clock64() - t; }
        else mbar_wait_role(&sched_full[slot], sphase);
        const uint2 it = ld_cluster_u32x2(ring_addr + slot * 8);
        mbar_arrive_remote(sched_empty_addr + slot * 8 + ring_dep(it));
        if (++slot == kP2Ring) { slot = 0; sphase ^= 1; }
        const int kind = it.x & 0xff;
        if (kind == IT_END) break;
        const P2Layer& ly = p.layer[kind];
        const uint32_t idesc = make_idesc_bf16(kP2Rows, static_cast<uint32_t>(ly.block_n));
#if PBG_KB_PROBE
        const long long pr_t1 = clock64();
#endif
        if (tr) { const long long t = clock64(); mbar_wait_role(&tmem_empty[acc], acc_phase ^ 1); w_tmem += clock64() - t; }
        else mbar_wait_role(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
#if PBG_KB_PROBE
        const long long pr_t2 = clock64();
        pr_item += pr_t1 - pr_t0; pr_tmem += pr_t2 - pr_t1;
#endif
        if (tr && n_it < kTraceItems) tr[16 + 4 * n_it + 1] = clock64();   // this item's accumulator stage is free: MMA start
        ++n_it;
        const uint32_t d_tmem = tmem_base + acc * 256;
        for (int kb = 0; kb < ly.num_kb; ++kb) {
          if (tr) {
            const long long t = clock64(); mbar_wait_role(&full_bar[stage], phase); const long long t1 = clock64();
            w_full += t1 - t; ++n_kb;
            const long long lat = t1 - t_issue[stage];
            if (t1 - t > 64) { lat_sum += lat; lat_n += 1; if (lat > lat_max) lat_max = lat; }  // only when the MMA really waited
          } else mbar_wait_role(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * L::kStage);
          const uint64_t da = make_kmajor_sw128_desc(sa);
          const uint64_t db = make_kmajor_sw128_desc(sa + L::kA);
#pragma unroll
          for (int k = 0; k < kBlockK / kUmmaK; ++k) umma_bf16_pair(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
          umma_commit_pair(&empty_bar[stage], 3);
          if (++stage == kP2Stages) { stage = 0; phase ^= 1; }
        }
        umma_commit_pair(&tmem_full[acc], 3);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
#if PBG_KB_PROBE
        pr_clk[kind] += clock64() - pr_t2; pr_tiles[kind] += 1;
#endif
      }
#if PBG_KB_PROBE
      {
        const int n = atomicAdd(&g_probe_n, 1), npairs = static_cast<int>(gridDim.x) / 2, pair = static_cast<int>(blockIdx.x) / 2;
        if (n / npairs == 30 && (pair == 0 || pair == npairs / 2 || pair == npairs - 1))
          printf("probe pair %d of %d (M=%d): MMA thread lifetime %lld clk; waiting for an item %lld, for a free accumulator %lld; "
                 "k-block loops (tiles: clk per tile) G.L0 %d: %lld  D.L0 %d: %lld  G.L1 %d: %lld  D.L1 %d: %lld  G.L2 %d: %lld\n",
                 pair, npairs, p.M, clock64() - pr_begin, pr_item, pr_tmem,
                 pr_tiles[0], pr_tiles[0] ? pr_clk[0] / pr_tiles[0] : 0, pr_tiles[1], pr_tiles[1] ? pr_clk[1] / pr_tiles[1] : 0,
                 pr_tiles[2], pr_tiles[2] ? pr_clk[2] / pr_tiles[2] : 0, pr_tiles[3], pr_tiles[3] ? pr_clk[3] / pr_tiles[3] : 0,
                 pr_tiles[4], pr_tiles[4] ? pr_clk[4] / pr_tiles[4] : 0);
      }
#endif
      if (tr) { tr[3] = w_full; tr[4] = w_tmem; tr[6] = clock64(); tr[9] = n_kb; tr[15] = w_item; tr[237] = lat_sum; tr[238] = lat_n; tr[239] = lat_max; }
    }
    __syncwarp();
  } else {
    // ------------------------------------------------------------ epilogue + gather warps (both CTAs)
    const int wep = warp - kEpiWarp0;  // 0..7
    const int q = warp & 3;            // TMEM lane quarter this warp may read
    const int half = wep >> 2;         // which half of a tile's 64-column chunks this warp takes
    // staging tile of warp (q, half): tiles of one lane quarter are adjacent, so that its two warps can lay whole output
    // rows (both column halves) out contiguously for the mirror stores of the last generator layer
    uint8_t* st = smem + L::kStagingOff + (q * kP2Slots + half) * L::kStagingPerWarp;
    uint32_t acc = 0, acc_phase = 0, slot = 0, sphase = 0;
    long long w_acc = 0, busy = 0, ph_wr = 0, ph_ld = 0, ph_math = 0, ph_st = 0, ph_n = 0, ph_m1 = 0, ph_w2 = 0;
    int item_no = 0;
    const int row_in_blk = static_cast<int>(rank) * 128 + q * 32 + lane;   // this thread's row within the 256-row block
    // The gather: 4-row groups claimed from a counter (claimed, not statically assigned: like the tickets, nothing may
    // depend on CTAs of this launch that are not resident yet -- several launches may share the device, and whatever
    // subset of a launch's CTAs is running has to be able to finish the pass on its own).  A warp gathers whenever it
    // would otherwise wait -- for a ring item, for an accumulator -- so only the first groups sit in front of the
    // first tiles; the counter hands the groups out in row order, which is the order the tiles need them in.
    bool more_groups = true;
    int pend_rb = -1;   // FASTG: row block of the group whose bulk stores are committed but not yet waited for
    auto gather_flush = [&]() {
      if (pend_rb >= 0) {
        if (lane == 0) { tma_store_wait<0>(); if (!p.gather_ahead) red_relaxed_gpu_add(p.ready + DEP_X * p.rb_cap + pend_rb, 1); }
        __syncwarp();
        pend_rb = -1;
      }
    };
    auto gather_one = [&]() {   // warp-uniform; false once every group has been claimed
      int g = 0;
      if (lane == 0) g = atomicAdd(&p.sched->p0_next, 1);
      g = __shfl_sync(0xffffffffu, g, 0);
      if (g >= p.phase0_groups) { more_groups = false; return; }
      if (tr && threadIdx.x == kTraceThread) tr[249] = clock64();
      if (FASTG) {
        p2_gather_group_bulk(p.gather, g, lane, st, gather_flush, p.gather_ahead != 0);
        if (tr && threadIdx.x == kTraceThread) tr[250] = clock64();
        pend_rb = static_cast<int>(g / kP2GroupsPerBlock);   // completed by the next group, or by gather_flush()
        if (!p.gather_defer) gather_flush();                 // PBG_GATHER_DEFER=0: complete every group at once
      } else {
        pass_gather_group<2>(p.gather, g, lane);
        if (tr && threadIdx.x == kTraceThread) tr[250] = clock64();
        if (!p.gather_ahead) p2_arrive(p, DEP_X, g / kP2GroupsPerBlock, lane, false);
        else __syncwarp();
      }
    };
    if (!p.gather_ahead) {
      gather_one();   // everybody starts with one group: nothing else can be ready yet
      gather_flush(); // ... and the first tiles wait for exactly these groups: no deferral for the first round
    }
    bool bias_ok = !BIASS;
    long long pf_wait = 0, pf_total = 0, pf_n = 0;
    // generator output rows of the previous PEPI_TANH tile may still be leaving through the quarter's two staging tiles
    bool pair_pending = false;
    auto pair_settle = [&]() {   // uniform over the quarter's two warps (both walk the same items)
      if (pair_pending) {
        if (half == 0 && lane == 0) tma_store_wait_read<0>();
        asm volatile("bar.sync %0, 64;" ::"r"(5 + q) : "memory");
        pair_pending = false;
      }
    };
    for (;;) {
      pair_settle();
      while (more_groups && !__all_sync(0xffffffffu, mbar_test_wait(&sched_full[slot], sphase))) gather_one();
      gather_flush();   // nothing may block, or touch the staging tile, with a group's arrival still owed
      mbar_wait(&sched_full[slot], sphase);
      const uint2 it = ld_cluster_u32x2(ring_addr + slot * 8);
      __syncwarp();
      if (lane == 0) mbar_arrive_remote(sched_empty_addr + slot * 8 + ring_dep(it));
      if (++slot == kP2Ring) { slot = 0; sphase ^= 1; }
      const int kind = it.x & 0xff;
      if (kind == IT_END) break;
      // idle until this item's accumulator is ready: gather (the staging tile is free between tiles)
      while (more_groups && !__all_sync(0xffffffffu, mbar_test_wait(&tmem_full[acc], acc_phase))) gather_one();
      gather_flush();
      if (tr && threadIdx.x == kTraceThread && tr[5] == 0) tr[5] = clock64();
      if (!bias_ok) { mbar_wait(bias_bar, 0); bias_ok = true; }  // the bias bulk copies issued in the prologue have landed
      const int n_blk = (it.x >> 8) & 0xff;
      const int rb = static_cast<int>(it.y);
      long long* ti = (tr && threadIdx.x == kTraceThread && item_no < kTraceItems) ? tr + 16 + 4 * item_no : nullptr;
      ++item_no;
      const P2Layer& ly = p.layer[kind];
      const long long grow = static_cast<long long>(rb) * kP2Rows + row_in_blk;
      const bool row_ok = grow < p.M;
      const int n0 = n_blk * ly.block_n;
      const int n_chunks = ly.block_n >> 6;   // 64-column chunks per tile; this warp takes c = half, half + 2, ...
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * 256;

      // PEPI_TANH prefetch (before the accumulator wait, i.e. behind the tile's MMA time): tail index, then the tail
      // values of this warp's first chunk -- columns 0..31 into the staging tile, columns 32..63 kept in registers
      const bool want_cos = ly.epi == PEPI_TANH && p.cosine != nullptr;
      unsigned long long trow_bits = 0ull;
      float4 tv2[8];
      if (want_cos) {
        const float* trow = nullptr;
        if (row_ok) {
          if (p.tail_idx != nullptr) {
            long long tid = p.tail_idx[grow * p.tail_stride];
            if (tid < 0) tid += p.n_ent;                  // same wrap as the gather
            tid = (tid < 0 || tid >= p.n_ent) ? 0 : tid;  // the gather has flagged it (tails are checked whenever given)
            trow = p.tail_tab + tid * p.n_valid;
          } else {
            trow = p.tail_tab + grow * p.n_valid;         // staged request: tail rows in request order
          }
        }
        trow_bits = reinterpret_cast<unsigned long long>(trow);
        if (half < n_chunks) {
          float4 tv1[8];
          p2_tail_load(tv1, trow_bits, n0 + half * 64, p.n_valid, lane);
          p2_tail_load(tv2, trow_bits, n0 + half * 64 + 32, p.n_valid, lane);
          p2_tail_stage(st, tv1, lane);
        }
      }
      {
        const long long t = (tr && lane == 0) ? clock64() : 0;
        mbar_wait(&tmem_full[acc], acc_phase);
        if (tr && lane == 0) { w_acc += clock64() - t; }
        if (ti) ti[2] = clock64();
      }
      const long long t_busy0 = (tr && lane == 0) ? clock64() : 0;
      tc_fence_after();

      if (ly.epi == PEPI_STORE) {
        // ---- bias + LeakyReLU -> bf16 -> swizzled staging tile -> global (TMA store, or transposed st.global)
        const bool tp = tr && threadIdx.x == kTraceThread;
        long long tq0 = 0, tq1 = 0, tq2 = 0, tq3 = 0, tq4 = 0, tq5 = 0, tq6 = 0;
        const float slope = p.slope;
        const float* const bias_tile = (BIASS ? sbias + ly.bias_off : ly.bias) + n0;
        const int row0 = rb * kP2Rows + static_cast<int>(rank) * 128 + q * 32;
        // 32-column TMEM loads, software pipelined: the next load is in flight while the previous one is converted
        uint32_t va[32], vb[32];
        if (half < n_chunks) tmem_ld_32x32_ptr(taddr + half * 64, va);
        for (int c = half; c < n_chunks; c += kP2Slots) {
          if (tp) tq0 = clock64();
          const float4* b4 = reinterpret_cast<const float4*>(bias_tile + c * 64);
          if (tp) tq1 = clock64();
          uint8_t* sbuf = st;
          tmem_ld_wait();
          tmem_ld_32x32_ptr(taddr + c * 64 + 32, vb);
          if (tp) tq2 = clock64();
          {
            float4 bq[8];
#pragma unroll
            for (int t = 0; t < 8; ++t) bq[t] = b4[t];
            uint4 w[4];
#pragma unroll
            for (int t = 0; t < 4; ++t) {
              const float4 ba = bq[2 * t], bb = bq[2 * t + 1];
              w[t].x = bias_leaky_pack(va[8 * t + 0], va[8 * t + 1], ba.x, ba.y, slope);
              w[t].y = bias_leaky_pack(va[8 * t + 2], va[8 * t + 3], ba.z, ba.w, slope);
              w[t].z = bias_leaky_pack(va[8 * t + 4], va[8 * t + 5], bb.x, bb.y, slope);
              w[t].w = bias_leaky_pack(va[8 * t + 6], va[8 * t + 7], bb.z, bb.w, slope);
            }
            // the staging tile is free once the previous chunk's bulk store has read it (hidden behind the math above)
            if (lane == 0) tma_store_wait_read<0>();
            __syncwarp();
#pragma unroll
            for (int t = 0; t < 4; ++t) *reinterpret_cast<uint4*>(sbuf + lane * 128 + ((t ^ (lane & 7)) << 4)) = w[t];
          }
          float4 bq[8];
#pragma unroll
          for (int t = 0; t < 8; ++t) bq[t] = b4[8 + t];   // in flight across the TMEM wait
          if (tp) tq5 = clock64();
          tmem_ld_wait();
          if (tp) tq6 = clock64();
          if (c + kP2Slots < n_chunks) {
            tmem_ld_32x32_ptr(taddr + (c + kP2Slots) * 64, va);
          } else {  // this warp's last read of the accumulator stage
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_remote(lead_tmem_empty + acc * 8);
          }
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const float4 ba = bq[2 * t], bb = bq[2 * t + 1];
            uint4 w;
            w.x = bias_leaky_pack(vb[8 * t + 0], vb[8 * t + 1], ba.x, ba.y, slope);
            w.y = bias_leaky_pack(vb[8 * t + 2], vb[8 * t + 3], ba.z, ba.w, slope);
            w.z = bias_leaky_pack(vb[8 * t + 4], vb[8 * t + 5], bb.x, bb.y, slope);
            w.w = bias_leaky_pack(vb[8 * t + 6], vb[8 * t + 7], bb.z, bb.w, slope);
            *reinterpret_cast<uint4*>(sbuf + lane * 128 + (((4 + t) ^ (lane & 7)) << 4)) = w;
          }
          if (tp) tq3 = clock64();
          fence_proxy_async_smem();  // generic-proxy writes of the staging tile -> visible to the bulk store
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(&p.tm_o[kind], sbuf, n0 + c * 64, row0);
            tma_store_commit();
          }
          if (tp) { tq4 = clock64(); ph_wr += tq1 - tq0; ph_ld += tq2 - tq1; ph_math += tq3 - tq2; ph_st += tq4 - tq3; ph_n += 1; ph_m1 += tq5 - tq2; ph_w2 += tq6 - tq5; }
        }
        if (half >= n_chunks) {  // narrow tile: this warp had no chunk, still has to release the accumulator
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_remote(lead_tmem_empty + acc * 8);
        }
        // publish the tile: its bulk stores must have completed (a few hundred clocks: the hand-off latency is on the
        // critical path of a small batch, so this is not deferred)
        {
          const long long t0 = (tr && threadIdx.x == kTraceThread) ? clock64() : 0;
          p2_arrive(p, ly.out_kind, rb, lane, true, (tr && threadIdx.x == kTraceThread) ? &pf_wait : nullptr);
          if (tr && threadIdx.x == kTraceThread) { pf_total += clock64() - t0; pf_n += 1; }
        }
        // G layer 1, first tile of the row block: every G L0 tile of the block has been published, so the block's gathered
        // rows are dead (when they are this pass's to drop: dead_xg)
        if (p.discard && kind == IT_G_L1 && n_blk == 0 && p.dead_xg != nullptr)
          p2_discard(static_cast<const char*>(p.dead_xg) + static_cast<size_t>(rb) * kP2Rows * p.dead_ldg * 2,
                     static_cast<size_t>(kP2Rows) * p.dead_ldg * 2, static_cast<int>(rank) * kP2Epi + wep, kP2WarpsPerPair, lane);
      } else if (ly.epi == PEPI_ROWDOT) {
        // ---- bias + LeakyReLU, dotted with the final [H/2 -> 1] weight; one partial per 64 columns, summed in a
        //      fixed order by the last warp to arrive for this row block
        const float slope = p.slope;
        float* part = p.part_d + (static_cast<size_t>(rb) * p.slots_d) * kP2Rows;
        for (int c = half; c < n_chunks; c += kP2Slots) {
          uint32_t v[64];
          tmem_ld_32x32_ptr(taddr + c * 64, v);
          tmem_ld_32x32_ptr(taddr + c * 64 + 32, v + 32);
          const float4* b4 = reinterpret_cast<const float4*>((BIASS ? sbias + ly.bias_off : ly.bias) + n0 + c * 64);
          const float4* w4 = reinterpret_cast<const float4*>((BIASS ? sbias + p.w3_off : p.w3) + n0 + c * 64);
          tmem_ld_wait();
          if (c + kP2Slots >= n_chunks) {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_remote(lead_tmem_empty + acc * 8);
          }
          float rowdot = 0.f;
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float4 b = b4[j], w = w4[j];
            rowdot = fmaf(leaky_max(__uint_as_float(v[4 * j + 0]) + b.x, slope), w.x, rowdot);
            rowdot = fmaf(leaky_max(__uint_as_float(v[4 * j + 1]) + b.y, slope), w.y, rowdot);
            rowdot = fmaf(leaky_max(__uint_as_float(v[4 * j + 2]) + b.z, slope), w.z, rowdot);
            rowdot = fmaf(leaky_max(__uint_as_float(v[4 * j + 3]) + b.w, slope), w.w, rowdot);
          }
          part[((n0 >> 6) + c) * kP2Rows + row_in_blk] = rowdot;
        }
        if (half >= n_chunks) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_remote(lead_tmem_empty + acc * 8);
        }
        // first tile of the row block: every D L0 tile of the block has been published -> its gathered rows are dead
        if (p.discard && n_blk == 0 && p.dead_xd != nullptr)
          p2_discard(static_cast<const char*>(p.dead_xd) + static_cast<size_t>(rb) * kP2Rows * p.dead_ldd * 2,
                     static_cast<size_t>(kP2Rows) * p.dead_ldd * 2, static_cast<int>(rank) * kP2Epi + wep, kP2WarpsPerPair, lane);
        const int old = warp_publish_fetch(p.fin + FIN_D * p.rb_cap + rb, lane);
        if (old == ly.n_tiles * kP2WarpsPerPair - 1) {
          fence_acq_rel_gpu();
          __syncwarp();
          // every D L1 tile of the block is done (its MMAs completed before its warps arrived here): the block's D L0
          // activations are dead
          if (p.discard)
            p2_discard(reinterpret_cast<const char*>(p.layer[IT_D_L0].out) + static_cast<size_t>(rb) * kP2Rows * p.layer[IT_D_L0].ldo * 2,
                       static_cast<size_t>(kP2Rows) * p.layer[IT_D_L0].ldo * 2, 0, 1, lane);
          // 8 rows per lane; all loads of a row group in flight together, summed in slot order
          float s[kP2Rows / 32];
#pragma unroll
          for (int j = 0; j < kP2Rows / 32; ++j) s[j] = 0.f;
          for (int k = 0; k < p.slots_d; ++k) {
            float x[kP2Rows / 32];
#pragma unroll
            for (int j = 0; j < kP2Rows / 32; ++j) x[j] = __ldcg(part + k * kP2Rows + j * 32 + lane);
#pragma unroll
            for (int j = 0; j < kP2Rows / 32; ++j) s[j] += x[j];
          }
#pragma unroll
          for (int j = 0; j < kP2Rows / 32; ++j) {
            const long long gr = static_cast<long long>(rb) * kP2Rows + j * 32 + lane;
            if (gr < p.M) {
              const float logit = s[j] + p.b3;
              const float prob = 1.f / (1.f + __expf(-logit));
              p.logits[gr] = logit;
              if (p.probs != nullptr) p.probs[gr] = prob;
              for (int mi = 0; mi < p.n_mirror; ++mi) {
                p.mir_logits[mi][gr] = logit;
                if (p.mir_probs[mi] != nullptr) p.mir_probs[mi][gr] = prob;
              }
              if (p.mc_logits != nullptr) multimem_st_f32(p.mc_logits + gr, logit);
              if (p.mc_probs != nullptr) multimem_st_f32(p.mc_probs + gr, prob);
            }
          }
        }
      } else {
        // ---- PEPI_TANH: bias + tanh -> generator output (fp32 / bf16), optional cosine vs the tail embedding
        const bool tpt = tr && threadIdx.x == kTraceThread;
        if (tpt) tr[232] = clock64();
        const bool want_out = p.gen_out != nullptr;
        const bool in_cta = ly.n_tiles == 1 && n_chunks == 2;  // the whole output row lives in this quarter's two warps
        float* part = p.part_g + (static_cast<size_t>(rb) * p.slots_g) * 3 * kP2Rows;
        for (int c = half; c < n_chunks; c += kP2Slots) {
          const int col0 = n0 + c * 64;
          if (want_cos && c != half) {  // later chunks of a wide tile: fetch their tail values now
            float4 tv1[8];
            p2_tail_load(tv1, trow_bits, col0, p.n_valid, lane);
            p2_tail_load(tv2, trow_bits, col0 + 32, p.n_valid, lane);
            p2_tail_stage(st, tv1, lane);
          }
          uint32_t v[64];
          tmem_ld_32x32_ptr(taddr + c * 64, v);
          tmem_ld_32x32_ptr(taddr + c * 64 + 32, v + 32);
          const float4* b4 = reinterpret_cast<const float4*>((BIASS ? sbias + ly.bias_off : ly.bias) + col0);
          tmem_ld_wait();
          if (c + kP2Slots >= n_chunks) {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_remote(lead_tmem_empty + acc * 8);
          }
          float* f = reinterpret_cast<float*>(v);
          if (tpt) tr[233] = clock64();
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float4 b = b4[j];
            f[4 * j + 0] = tanh_fast(f[4 * j + 0] + b.x);
            f[4 * j + 1] = tanh_fast(f[4 * j + 1] + b.y);
            f[4 * j + 2] = tanh_fast(f[4 * j + 2] + b.z);
            f[4 * j + 3] = tanh_fast(f[4 * j + 3] + b.w);
          }
          if (tpt) tr[234] = clock64();
          if (want_cos) {
            // columns 0..31 are in the staging tile (one row per lane); then columns 32..63 take their place
            float cs_dot = 0.f, cs_pp = 0.f, cs_tt = 0.f;
            p2_tail_dot(st, f, col0, p.n_valid, lane, cs_dot, cs_pp, cs_tt);
            p2_tail_stage(st, tv2, lane);
            p2_tail_dot(st, f + 32, col0 + 32, p.n_valid, lane, cs_dot, cs_pp, cs_tt);
            if (tpt) tr[245] = clock64();
            if (in_cta) {
              // the two warps of this lane quarter hold the row's two halves: the upper one hands its sums over
              // through shared memory, the lower one finishes (fixed order: columns 0..63 + columns 64..127)
              float* xq = xchg + (q * 32 + lane) * 3;
              if (half == 1) { xq[0] = cs_dot; xq[1] = cs_pp; xq[2] = cs_tt; }
              asm volatile("bar.sync %0, 64;" ::"r"(1 + q) : "memory");
              if (tpt) tr[255] = clock64();
              if (half == 0) {
                const float d = cs_dot + xq[0], pp = cs_pp + xq[1], tt = cs_tt + xq[2];
                // F.cosine_similarity(pred, t, dim=1), eps = 1e-8 on each norm (pro_b_gan_infer.py:202)
                if (row_ok) {
                  const float cs = d / (fmaxf(sqrtf(pp), 1e-8f) * fmaxf(sqrtf(tt), 1e-8f));
                  p.cosine[grow] = cs;
                  for (int mi = 0; mi < p.n_mirror; ++mi) p.mir_cos[mi][grow] = cs;
                  if (p.mc_cos != nullptr) multimem_st_f32(p.mc_cos + grow, cs);
                }
              }
              asm volatile("bar.sync %0, 64;" ::"r"(1 + q) : "memory");  // the slot may be rewritten after this
            } else if (col0 < p.n_valid) {
              float* mine = part + (col0 >> 6) * 3 * kP2Rows;  // one partial triple per 64-column chunk
              mine[row_in_blk] = cs_dot;
              mine[kP2Rows + row_in_blk] = cs_pp;
              mine[2 * kP2Rows + row_in_blk] = cs_tt;
            }
          }
          if (tpt) tr[235] = clock64();
          // Common case (bf16 rows of 128 columns: this quarter's two warps hold 32 whole, consecutive rows): the rows
          // are laid out in the two warps' staging tiles and leave as ONE 8 KB bulk store to the caller's buffer and
          // one per mirror.  Otherwise: 16-byte stores from registers to the caller's buffer, and for mirrors (peer
          // GPUs over NVLink, where 16-byte stores would cross the link as 16-byte packets) one 128-byte bulk store
          // per lane and mirror.
          const bool bulk_mirror = p.n_mirror > 0 && (p.n_valid & 63) == 0;
          const bool pair_out = want_out && in_cta && !p.out_f32 && p.n_valid == 128 && p.ld_gen == 128;
          if (want_out && row_ok && !pair_out) {
            // one row per lane, 16-byte stores (2 MB for a 4096-row pass: not worth a transpose through shared memory)
            // the caller's own buffer: 16-byte stores straight from registers; mirrors (peer GPUs over NVLink): the row
            // segment goes through this lane's 128 bytes of the staging tile and out as one 128-byte bulk store per
            // mirror -- 16-byte stores would cross NVLink as 16-byte packets
            for (int mi = -1; mi < (bulk_mirror ? 0 : p.n_mirror); ++mi) {
              void* base = mi < 0 ? p.gen_out : p.mir_gen[mi];
              if (p.out_f32) {
                float* orow = static_cast<float*>(base) + grow * p.ld_gen + col0;
#pragma unroll
                for (int t = 0; t < 16; ++t)
                  if (col0 + t * 4 < p.n_valid)
                    *reinterpret_cast<float4*>(orow + t * 4) = make_float4(f[4 * t], f[4 * t + 1], f[4 * t + 2], f[4 * t + 3]);
              } else {
                __nv_bfloat16* orow = static_cast<__nv_bfloat16*>(base) + grow * p.ld_gen + col0;
#pragma unroll
                for (int t = 0; t < 8; ++t) {
                  uint4 w;
                  w.x = pack_bf16x2(f[8 * t + 0], f[8 * t + 1]);
                  w.y = pack_bf16x2(f[8 * t + 2], f[8 * t + 3]);
                  w.z = pack_bf16x2(f[8 * t + 4], f[8 * t + 5]);
                  w.w = pack_bf16x2(f[8 * t + 6], f[8 * t + 7]);
                  if (col0 + t * 8 < p.n_valid) *reinterpret_cast<uint4*>(orow + t * 8) = w;
                }
              }
            }
            if (p.mc_gen != nullptr) {   // uncommon shapes (fp32 output, E != 128): 16-byte multicast stores from registers
              if (p.out_f32) {
                char* orow = static_cast<char*>(p.mc_gen) + (static_cast<size_t>(grow) * p.ld_gen + col0) * 4;
#pragma unroll
                for (int t = 0; t < 16; ++t)
                  if (col0 + t * 4 < p.n_valid)
                    multimem_st_v4(orow + t * 16, make_uint4(__float_as_uint(f[4 * t]), __float_as_uint(f[4 * t + 1]),
                                                             __float_as_uint(f[4 * t + 2]), __float_as_uint(f[4 * t + 3])));
              } else {
                char* orow = static_cast<char*>(p.mc_gen) + (static_cast<size_t>(grow) * p.ld_gen + col0) * 2;
#pragma unroll
                for (int t = 0; t < 8; ++t) {
                  uint4 w;
                  w.x = pack_bf16x2(f[8 * t + 0], f[8 * t + 1]);
                  w.y = pack_bf16x2(f[8 * t + 2], f[8 * t + 3]);
                  w.z = pack_bf16x2(f[8 * t + 4], f[8 * t + 5]);
                  w.w = pack_bf16x2(f[8 * t + 6], f[8 * t + 7]);
                  if (col0 + t * 8 < p.n_valid) multimem_st_v4(orow + t * 16, w);
                }
              }
            }
            // bulk_mirror implies embed_dim % 64 == 0, so a chunk is wholly valid or wholly padding; a padding chunk
            // (E = 64, 192, 320, ...) has nothing to mirror, and its 128 bytes would land on the next row
            if (bulk_mirror && col0 < p.n_valid) {
              uint8_t* myrow = st + lane * 128;   // only this lane writes and (through its bulk stores) reads it
              const int rounds = p.out_f32 ? 2 : 1;
              for (int rd = 0; rd < rounds; ++rd) {
                tma_store_wait_read<0>();         // this lane's earlier bulk stores have read the row
                if (p.out_f32) {
#pragma unroll
                  for (int t = 0; t < 8; ++t)
                    *reinterpret_cast<float4*>(myrow + t * 16) =
                        make_float4(f[32 * rd + 4 * t], f[32 * rd + 4 * t + 1], f[32 * rd + 4 * t + 2], f[32 * rd + 4 * t + 3]);
                } else {
#pragma unroll
                  for (int t = 0; t < 8; ++t) {
                    uint4 w;
                    w.x = pack_bf16x2(f[8 * t + 0], f[8 * t + 1]);
                    w.y = pack_bf16x2(f[8 * t + 2], f[8 * t + 3]);
                    w.z = pack_bf16x2(f[8 * t + 4], f[8 * t + 5]);
                    w.w = pack_bf16x2(f[8 * t + 6], f[8 * t + 7]);
                    *reinterpret_cast<uint4*>(myrow + t * 16) = w;
                  }
                }
                fence_proxy_async_smem();
                const size_t es = p.out_f32 ? 4 : 2;
                const size_t byte_off = (static_cast<size_t>(grow) * p.ld_gen + col0) * es + static_cast<size_t>(rd) * 128;
                for (int mi = 0; mi < p.n_mirror; ++mi) bulk_store_1d(static_cast<char*>(p.mir_gen[mi]) + byte_off, myrow, 128);
                tma_store_commit();
              }
            }
          }
          if (pair_out) {                     // (uniform over the quarter's two warps)
            uint8_t* region = smem + L::kStagingOff + q * kP2Slots * L::kStagingPerWarp;   // the first two warps' tiles: 32 rows x 256 B
            asm volatile("bar.sync %0, 64;" ::"r"(5 + q) : "memory");   // both warps are done with their own tiles
#pragma unroll
            for (int t = 0; t < 8; ++t) {
              uint4 w;
              w.x = pack_bf16x2(f[8 * t + 0], f[8 * t + 1]);
              w.y = pack_bf16x2(f[8 * t + 2], f[8 * t + 3]);
              w.z = pack_bf16x2(f[8 * t + 4], f[8 * t + 5]);
              w.w = pack_bf16x2(f[8 * t + 6], f[8 * t + 7]);
              *reinterpret_cast<uint4*>(region + lane * 256 + half * 128 + t * 16) = w;
            }
            fence_proxy_async_smem();
            asm volatile("bar.sync %0, 64;" ::"r"(5 + q) : "memory");   // the rows are complete
            if (half == 0 && lane == 0) {
              const long long row0 = grow - lane;
              const long long nrows = min(32ll, p.M - row0);
              if (nrows > 0) {
                bulk_store_1d(static_cast<char*>(p.gen_out) + row0 * 256, region, static_cast<uint32_t>(nrows * 256));
                for (int mi = 0; mi < p.n_mirror; ++mi)
                  bulk_store_1d(static_cast<char*>(p.mir_gen[mi]) + row0 * 256, region, static_cast<uint32_t>(nrows * 256));
                tma_store_commit();
              }
            }
            if (p.mc_gen != nullptr) {
              // multi-GPU: the same 8 KB leave once through the multicast address, 16 bytes per thread and store, 512
              // contiguous bytes per warp instruction; NVSwitch writes them into every GPU's copy of the buffer
              const long long row0 = grow - lane;
              const int nbytes = static_cast<int>(min(32ll, p.M - row0)) * 256;
              char* dst = static_cast<char*>(p.mc_gen) + row0 * 256;
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const int off = (i * 64 + half * 32 + lane) * 16;
                if (off < nbytes) multimem_st_v4(dst + off, *reinterpret_cast<const uint4*>(region + off));
              }
            }
            // The bulk engine is still reading the region (one 8 KB read per destination: the caller's buffer and up to
            // seven mirrors over NVLink).  Nobody waits for that here: pair_settle() does, right before the quarter's
            // staging tiles are next written -- normally many thousand clocks later, or never (last item of the pass).
            pair_pending = true;
          }
          if (want_out && p.n_mirror > 0 && !pair_out) {   // (warp-uniform) the staging tile is free again when every lane's stores have read it
            tma_store_wait_read<0>();
            __syncwarp();
          }
        }
        if (half >= n_chunks) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_remote(lead_tmem_empty + acc * 8);
        }
        // this tile's MMAs have read the block's G L1 activations, and every G L1 tile of the block was published before
        // this tile was (each after its own MMAs): with one G L2 tile per row block both activation blocks are dead
        if (p.discard && ly.n_tiles == 1) {
          const int part = static_cast<int>(rank) * kP2Epi + wep;
          p2_discard(reinterpret_cast<const char*>(p.layer[IT_G_L0].out) + static_cast<size_t>(rb) * kP2Rows * p.layer[IT_G_L0].ldo * 2,
                     static_cast<size_t>(kP2Rows) * p.layer[IT_G_L0].ldo * 2, part, kP2WarpsPerPair, lane);
          p2_discard(reinterpret_cast<const char*>(p.layer[IT_G_L1].out) + static_cast<size_t>(rb) * kP2Rows * p.layer[IT_G_L1].ldo * 2,
                     static_cast<size_t>(kP2Rows) * p.layer[IT_G_L1].ldo * 2, part, kP2WarpsPerPair, lane);
        }
        if (tpt) tr[236] = clock64();
        if (want_cos && !in_cta) {
          const int old = warp_publish_fetch(p.fin + FIN_G * p.rb_cap + rb, lane);
          if (old == ly.n_tiles * kP2WarpsPerPair - 1) {
            fence_acq_rel_gpu();
            __syncwarp();
            for (int r = lane; r < kP2Rows; r += 32) {
              const long long gr = static_cast<long long>(rb) * kP2Rows + r;
              float d = 0.f, pp = 0.f, tt = 0.f;
              for (int k = 0; k < p.slots_g; ++k) {
                d += __ldcg(part + (k * 3 + 0) * kP2Rows + r);
                pp += __ldcg(part + (k * 3 + 1) * kP2Rows + r);
                tt += __ldcg(part + (k * 3 + 2) * kP2Rows + r);
              }
              if (gr < p.M) {
                const float cs = d / (fmaxf(sqrtf(pp), 1e-8f) * fmaxf(sqrtf(tt), 1e-8f));
                p.cosine[gr] = cs;
                for (int mi = 0; mi < p.n_mirror; ++mi) p.mir_cos[mi][gr] = cs;
                if (p.mc_cos != nullptr) multimem_st_f32(p.mc_cos + gr, cs);
              }
            }
          }
        }
      }
      if (tr && lane == 0) busy += clock64() - t_busy0;
      if (ti) ti[3] = clock64();
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
    if (p.gather_ahead) {   // whatever is left of the next request's rows (claimed from the same counter by every warp)
      pair_settle();
      while (more_groups) gather_one();
      gather_flush();
    }
    // every lane: its bulk stores must have READ the staging tile before the CTA (and its shared memory) goes away; their
    // global / peer writes complete with the grid -- waiting for them here would put an NVLink round trip on every CTA's exit
    tma_store_wait_read<0>();
    if (tr && threadIdx.x == kTraceThread) {
      tr[7] = w_acc; tr[8] = clock64(); tr[10] = busy;
      tr[240] = ph_ld; tr[241] = ph_math; tr[242] = ph_st; tr[243] = ph_n; tr[244] = ph_wr;
      tr[251] = ph_m1; tr[252] = ph_w2;
      tr[246] = pf_wait; tr[247] = pf_total; tr[248] = pf_n;
    }
  }

  // teardown: neither CTA may exit while the other can still touch its shared memory / barriers / TMEM
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == kMmaWarp) {
    tc_fence_after();
    tmem_dealloc_pair<512>(tmem_base);
  }
  // the last CTA to finish re-arms the scheduler and zeroes the arrival counters for the next launch
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    p.sched->clk_ticks = clock64() - clk0[0];
    p.sched->clk_ns = static_cast<long long>(globaltimer_ns()) - clk0[1];
  }
  if (threadIdx.x == 0) {
    const int old = atomicAdd(&p.sched->done, 1);
    *last_flag = (old == static_cast<int>(gridDim.x) - 1);
  }
  __syncthreads();
  if (*last_flag) {
    for (int k = 0; k < DEP_KINDS; ++k)
      for (int i = threadIdx.x; i < p.nrb; i += blockDim.x) p.ready[k * p.rb_cap + i] = 0;
    for (int k = 0; k < FIN_KINDS; ++k)
      for (int i = threadIdx.x; i < p.nrb; i += blockDim.x) p.fin[k * p.rb_cap + i] = 0;
    if (threadIdx.x == 0) { p.sched->q_head = 0; p.sched->q_tail = 0; p.sched->p0_next = 0; p.sched->init = 0; p.sched->done = 0; }
    if (tr && threadIdx.x == 0) { tr[13] = clock64(); tr[253] = static_cast<long long>(globaltimer_ns()); }
  }
}

}  // namespace pbg
