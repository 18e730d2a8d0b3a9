// pbg.cu -- libpbg_b200.so: context, weight ingest, workspaces, TMA descriptors and the launch sequence behind
// the C ABI declared in include/pbg.h.  Device code lives in gather.cuh / pass2_kernel.cuh / topk_kernel.cuh / gemm_f32.cuh /
// latent.cuh.
//
// HBM layout per ctx (sized lazily to the largest batch chunk seen, <= kMaxChunk rows):
//   weights   : fp32 [out,in] + bias (parity mode) and bf16 [out_p, in_p] zero-padded to the tile grid + padded bias
//   bf16 mode : xg0 [rows, Kg0p]  xd0 [rows, Kd0p]  bufA [rows, Hmax]  bufB [rows, Hmax]  bufD [rows, Hdp]  (bf16,
//               K-major, the A operands of the next GEMM, each with a SWIZZLE_128B CUtensorMap of box 128 x 64); two
//               staging slots (xg0, xd0, fp32 tail rows) for requests gathered ahead of their pass
//   fp32 mode : xg0, xd0, bufA, bufB in fp32
// bf16 mode, one launch: G: xg0 -> bufA -> bufB -> out.   D: xd0 -> bufD -> (logit, prob); a row block of these buffers is
// dropped from L2 (discard.global.L2) once its consumer layer is done with it.  fp32 mode, a launch per layer:
// G: xg0 -> bufA -> bufB -> out.   D: xd0 -> bufA -> bufB -> (logit, prob).   One stream at a time per ctx.
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <map>
#include <tuple>
#include <new>
#include <string>
#include <vector>

#include "../../include/pbg.h"
#include "gather.cuh"
#include "gemm_f32.cuh"
#include "tc_common.cuh"
#include "pass_common.cuh"
#include "pass2_kernel.cuh"
#include "topk_kernel.cuh"
#include "index_rows.cuh"
#include "json_out.cuh"
#include "latent.cuh"

using namespace pbg;

namespace {

constexpr long long kMaxChunk = 65536;  // rows processed per launch sequence (bounds the workspaces)
constexpr int kPartSlotsG = 16;  // generator cosine partials per row: one per 32 output columns (E <= 512)
constexpr int kPartSlotsD = 64;  // discriminator dot partials per row: one per 64 columns of H/2 (H <= 8192)

inline int round_up(int v, int m) { return (v + m - 1) / m * m; }

struct Linear {
  int n = 0, k = 0;    // logical [out, in]
  int np = 0, kp = 0;  // padded to the tensor-core tile grid
  float* w_f32 = nullptr;
  float* b_f32 = nullptr;
  __nv_bfloat16* w_bf16 = nullptr;
  float* b_pad = nullptr;
  CUtensorMap tmap_w128;  // box 64 x 128 (finer tiles for small batches; one CTA's half of a 256-wide pair tile)
  CUtensorMap tmap_w64;   // box 64 x 64  (one CTA's half of a 128-wide pair tile)
};

struct Workspace {
  long long rows = 0;
  void *xg0 = nullptr, *xd0 = nullptr, *bufA = nullptr, *bufB = nullptr, *bufD = nullptr;
  CUtensorMap tm_xg0, tm_xd0, tm_bufA_g, tm_bufA_d, tm_bufB_g, tm_bufD_d;
  CUtensorMap tmo_bufA, tmo_bufB, tmo_bufD;  // store maps: box 64 x 32 (one epilogue warp's chunk)
  // fused pass kernel state (bf16 mode): arrival counters, scheduler, row-reduction partials
  int mb_cap = 0;
  int* ready = nullptr;   // [DEP_KINDS][mb_cap]
  int* fin = nullptr;     // [FIN_KINDS][mb_cap]
  PassSched* sched = nullptr;
  float* part_g = nullptr;  // [mb_cap][4][3][128]
  float* part_d = nullptr;  // [mb_cap][2 * max n_tiles][128]
};

// entity scoring + top-k (pbg_topk_prepare / pbg_topk)
struct TopkState {
  const float* table = nullptr; long long N = 0, n_pad = 0;
  __nv_bfloat16* tn = nullptr; float* inv_t = nullptr; CUtensorMap tm_t;
  long long q_cap = 0; __nv_bfloat16* qn = nullptr; float* inv_q = nullptr; CUtensorMap tm_q;
  size_t cand_cap = 0; unsigned* cand_grp = nullptr; unsigned* cand_mask = nullptr; int* cand_cnt = nullptr;   // [rows][lists][kTkCand]
  size_t samp_cap = 0; int* samp_keys = nullptr;   // [rows][sample lists][kTkKeys]
  float* tau = nullptr; int* flag = nullptr;       // [q_cap]
  long long last_rows = 0; bool last_filtered = false;   // the last chunk pbg_topk ran (pbg_topk_last_flagged)
  size_t score_cap = 0; float* score_buf = nullptr;  // general path: exact scores of a chunk of rows [rows, N]
};

// One staged request (pbg_stage_triplets): the first-layer operands of the pass, gathered + concatenated + cast by the
// staging kernel on the caller's ingest stream while the previous request's pass is still running.
struct StageSlot {
  long long cap = 0;  // rows allocated
  void *xg0 = nullptr, *xd0 = nullptr;
  float* xt = nullptr;  // fp32 tail rows [cap, E] for the cosine epilogue
  float* z = nullptr;   // fp32 latents [cap, Z] drawn from the ctx's latent stream when the request brings none
  CUtensorMap tm_xg0, tm_xd0;
  long long B = -1;     // rows of the staged request (-1: nothing staged)
  bool has_g = false, has_d = false;
  bool has_xt = false;  // xt holds the tail rows (staging kernel); otherwise the cosine epilogue indexes the table itself
  const float* node_emb = nullptr; long long N = 0; const long long* tails = nullptr;   // ... through these (stride 3)
};

thread_local std::string g_create_error;

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

}  // namespace

struct pbg_ctx {
  pbg_dims dims{};
  int num_sms = 0;
  int max_threads_sm = 0;   // with num_sms, sets torch's launch geometry that the latent draw reproduces
  bool g_loaded = false, d_loaded = false;
  int kg0 = 0, kg0p = 0, kd0 = 0, kd0p = 0, hgp = 0, hdp = 0, hd2 = 0, hmax = 0;
  Linear g[3], d[2];
  float* d_w3 = nullptr;      // [hd2] fp32
  float* d_w3_pad = nullptr;  // [hd2p]
  float d_b3 = 0.f;
  Workspace ws_bf16, ws_f32;
  StageSlot stage[2];
  int* err_flag = nullptr;       // device
  int* err_flag_host = nullptr;  // pinned
  cudaStream_t own_stream = nullptr;
  // device staging for the *_host entry point: ONE block [triplets | z | scores | logits | probs | gen_out], so that
  // host buffers the caller laid out the same way travel in one copy per direction
  long long host_cap = 0;
  char* st_block = nullptr;
  EncodeTiledFn encode = nullptr;
  TopkState tk;
  // latent stream (pbg_set_latent_stream): generator calls without z draw from Philox (lat_seed, lat_st->offset)
  bool lat_on = false;
  unsigned long long lat_seed = 0;
  LatentStream* lat_st = nullptr;   // device: the offset, advanced by each draw
  long long lat_cap = 0;            // rows of lat_z
  float* lat_z = nullptr;           // [lat_cap, Z] the drawn latents of the current chunk
  long long launches = 0;
  int launch_ctas = 0;  // pbg_set_launch_width; 0 = all SMs
  int discard = 1;      // pbg_set_workspace_discard (PBG_DISCARD sets the initial value)
  bool host_block = false;          // PBG_HOST_SYNC=block: the *_host entry points sleep on an event instead of spinning
  cudaEvent_t host_evt = nullptr;   // cudaEventBlockingSync
  int n_mirror = 0;     // pbg_set_result_mirrors
  void* mir_gen[kMaxMirrors] = {}; float* mir_cos[kMaxMirrors] = {}; float* mir_logits[kMaxMirrors] = {}; float* mir_probs[kMaxMirrors] = {};
  void* mc_gen = nullptr; float *mc_cos = nullptr, *mc_logits = nullptr, *mc_probs = nullptr;   // pbg_set_result_multicast
  bool profiling = false;
  long long* trace = nullptr;  // device, 16 slots x num_sms (pbg_debug_trace)
  struct ProfRec { cudaEvent_t a, b; int kind; };
  std::vector<ProfRec> prof;
  std::string err;
};

namespace {

int fail(pbg_ctx* c, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (c) c->err = buf; else g_create_error = buf;
  return code;
}

// Brackets one kernel launch with events when profiling is on (bench.py roofline), and counts it.
struct LaunchScope {
  pbg_ctx* c; cudaStream_t s; cudaEvent_t b = nullptr;
  LaunchScope(pbg_ctx* c_, int kind, cudaStream_t s_) : c(c_), s(s_) {
    c->launches += 1;
    if (c->profiling) {
      cudaEvent_t a;
      cudaEventCreate(&a); cudaEventCreate(&b);
      cudaEventRecord(a, s);
      c->prof.push_back({a, b, kind});
    }
  }
  ~LaunchScope() { if (b) cudaEventRecord(b, s); }
};

#define PBG_CUDA(c, expr)                                                                               \
  do {                                                                                                  \
    cudaError_t e_ = (expr);                                                                            \
    if (e_ != cudaSuccess) return fail((c), PBG_ERR_CUDA, "%s failed: %s", #expr, cudaGetErrorString(e_)); \
  } while (0)

#define PBG_TRY(expr)            \
  do {                           \
    int s_ = (expr);             \
    if (s_ != PBG_OK) return s_; \
  } while (0)

int make_tmap(pbg_ctx* c, CUtensorMap* tm, const void* base, long long rows, int cols, int box_rows) {
  // 2-D bf16 [rows, cols] row-major; box = box_rows x 64 elements (128 B inner = one swizzle row)
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(cols) * 2};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(kBlockK), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = c->encode(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(c, PBG_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) rows=%lld cols=%d", (int)r, rows, cols);
  return PBG_OK;
}

void free_linear(Linear& l) {
  cudaFree(l.w_f32); cudaFree(l.b_f32); cudaFree(l.w_bf16); cudaFree(l.b_pad);
  l = Linear{};
}

void free_ws(Workspace& w) {
  cudaFree(w.xg0); cudaFree(w.xd0); cudaFree(w.bufA); cudaFree(w.bufB); cudaFree(w.bufD);
  cudaFree(w.ready); cudaFree(w.fin); cudaFree(w.sched); cudaFree(w.part_g); cudaFree(w.part_d);
  w = Workspace{};
}

// Upload one Linear: fp32 copy for the parity mode, padded bf16 copy + TMA descriptors for the tensor-core mode.
int upload_linear(pbg_ctx* c, Linear& l, int n, int k, int kp, const float* w_host, const float* b_host) {
  free_linear(l);
  l.n = n; l.k = k; l.kp = kp;
  l.np = round_up(n, 128);
  PBG_CUDA(c, cudaMalloc(&l.w_f32, sizeof(float) * n * k));
  PBG_CUDA(c, cudaMalloc(&l.b_f32, sizeof(float) * n));
  PBG_CUDA(c, cudaMalloc(&l.w_bf16, sizeof(__nv_bfloat16) * (size_t)l.np * l.kp));
  PBG_CUDA(c, cudaMalloc(&l.b_pad, sizeof(float) * l.np));
  PBG_CUDA(c, cudaMemcpyAsync(l.w_f32, w_host, sizeof(float) * n * k, cudaMemcpyHostToDevice, c->own_stream));
  PBG_CUDA(c, cudaMemcpyAsync(l.b_f32, b_host, sizeof(float) * n, cudaMemcpyHostToDevice, c->own_stream));
  { LaunchScope ls(c, PBG_K_OTHER, c->own_stream);
    pack_bf16_kernel<<<c->num_sms * 4, 256, 0, c->own_stream>>>(l.w_f32, l.w_bf16, n, k, l.np, l.kp); }
  { LaunchScope ls(c, PBG_K_OTHER, c->own_stream);
    pad_f32_kernel<<<8, 256, 0, c->own_stream>>>(l.b_f32, l.b_pad, n, l.np); }
  PBG_CUDA(c, cudaGetLastError());
  PBG_CUDA(c, cudaStreamSynchronize(c->own_stream));
  PBG_TRY(make_tmap(c, &l.tmap_w128, l.w_bf16, l.np, l.kp, 128));
  return make_tmap(c, &l.tmap_w64, l.w_bf16, l.np, l.kp, 64);
}

// Growing a buffer means cudaDeviceSynchronize + cudaFree + cudaMalloc: illegal while `s` is being captured into a
// CUDA graph, and a device-wide stall for every other lane otherwise -- callers that care size everything up front
// with pbg_reserve().  Refuses inside a capture, otherwise waits until nothing may still be reading the old buffers.
int begin_growth(pbg_ctx* c, cudaStream_t s, const char* what) {
  cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(s, &st) == cudaSuccess && st != cudaStreamCaptureStatusNone)
    return fail(c, PBG_ERR_INVALID, "%s must grow while the stream is being captured: call pbg_reserve() first", what);
  PBG_CUDA(c, cudaDeviceSynchronize());
  return PBG_OK;
}

// Rows to allocate for `rows`: rounded up to a power of two in [1024, kMaxChunk], so that small calls do not keep
// reallocating.
long long pow2_cap(long long rows) {
  long long cap = 1024;
  while (cap < rows) cap *= 2;
  return std::min(cap, kMaxChunk);
}

// Replaces *p by a fresh allocation of `bytes`; *p is null if that fails.
template <class T>
int realloc_dev(pbg_ctx* c, T*& p, size_t bytes) {
  cudaFree(p); p = nullptr;
  PBG_CUDA(c, cudaMalloc(&p, bytes));
  return PBG_OK;
}

void free_stage(StageSlot& st) {
  cudaFree(st.xg0); cudaFree(st.xd0); cudaFree(st.xt); cudaFree(st.z);
  st = StageSlot{};
}

int ensure_ws(pbg_ctx* c, int prec, long long rows, cudaStream_t stream) {
  Workspace& w = prec == PBG_PREC_BF16 ? c->ws_bf16 : c->ws_f32;
  if (w.rows >= rows) return PBG_OK;
  PBG_TRY(begin_growth(c, stream, "the workspace"));
  const long long cap = pow2_cap(rows);
  free_ws(w);
  if (prec == PBG_PREC_BF16) {
    const size_t es = sizeof(__nv_bfloat16);
    PBG_CUDA(c, cudaMalloc(&w.xg0, es * cap * c->kg0p));
    PBG_CUDA(c, cudaMalloc(&w.xd0, es * cap * c->kd0p));
    PBG_CUDA(c, cudaMalloc(&w.bufA, es * cap * c->hmax));
    PBG_CUDA(c, cudaMalloc(&w.bufB, es * cap * c->hmax));
    PBG_CUDA(c, cudaMalloc(&w.bufD, es * cap * c->hdp));
    PBG_TRY(make_tmap(c, &w.tm_bufD_d, w.bufD, cap, c->hdp, kBlockM));
    PBG_TRY(make_tmap(c, &w.tmo_bufA, w.bufA, cap, c->hgp, 32));
    PBG_TRY(make_tmap(c, &w.tmo_bufB, w.bufB, cap, c->hgp, 32));
    PBG_TRY(make_tmap(c, &w.tmo_bufD, w.bufD, cap, c->hdp, 32));
    w.mb_cap = static_cast<int>(cap / kBlockM);
    PBG_CUDA(c, cudaMalloc(&w.ready, sizeof(int) * DEP_KINDS * w.mb_cap));
    PBG_CUDA(c, cudaMalloc(&w.fin, sizeof(int) * FIN_KINDS * w.mb_cap));
    PBG_CUDA(c, cudaMalloc(&w.sched, sizeof(PassSched)));
    PBG_CUDA(c, cudaMalloc(&w.part_g, sizeof(float) * w.mb_cap * kPartSlotsG * 3 * kBlockM));
    PBG_CUDA(c, cudaMalloc(&w.part_d, sizeof(float) * w.mb_cap * kPartSlotsD * kBlockM));
    PBG_CUDA(c, cudaMemset(w.ready, 0, sizeof(int) * DEP_KINDS * w.mb_cap));
    PBG_CUDA(c, cudaMemset(w.fin, 0, sizeof(int) * FIN_KINDS * w.mb_cap));
    PBG_CUDA(c, cudaMemset(w.sched, 0, sizeof(PassSched)));
    PBG_TRY(make_tmap(c, &w.tm_xg0, w.xg0, cap, c->kg0p, kBlockM));
    PBG_TRY(make_tmap(c, &w.tm_xd0, w.xd0, cap, c->kd0p, kBlockM));
    PBG_TRY(make_tmap(c, &w.tm_bufA_g, w.bufA, cap, c->hgp, kBlockM));
    PBG_TRY(make_tmap(c, &w.tm_bufA_d, w.bufA, cap, c->hdp, kBlockM));
    PBG_TRY(make_tmap(c, &w.tm_bufB_g, w.bufB, cap, c->hgp, kBlockM));
  } else {
    const size_t es = sizeof(float);
    const int hm = std::max(std::max(c->dims.g_hidden, c->dims.d_hidden), c->dims.embed_dim);
    PBG_CUDA(c, cudaMalloc(&w.xg0, es * cap * c->kg0));
    PBG_CUDA(c, cudaMalloc(&w.xd0, es * cap * c->kd0));
    PBG_CUDA(c, cudaMalloc(&w.bufA, es * cap * hm));
    PBG_CUDA(c, cudaMalloc(&w.bufB, es * cap * hm));
  }
  w.rows = cap;
  return PBG_OK;
}

int ensure_stage(pbg_ctx* c, StageSlot& st, long long rows, cudaStream_t stream) {
  if (st.cap >= rows) return PBG_OK;
  PBG_TRY(begin_growth(c, stream, "a staging slot"));
  const long long cap = pow2_cap(rows);
  free_stage(st);
  const size_t es = sizeof(__nv_bfloat16);
  PBG_CUDA(c, cudaMalloc(&st.xg0, es * cap * c->kg0p));
  PBG_CUDA(c, cudaMalloc(&st.xd0, es * cap * c->kd0p));
  PBG_CUDA(c, cudaMalloc(&st.xt, sizeof(float) * cap * c->dims.embed_dim));
  PBG_CUDA(c, cudaMalloc(&st.z, sizeof(float) * cap * c->dims.noise_dim));
  PBG_TRY(make_tmap(c, &st.tm_xg0, st.xg0, cap, c->kg0p, kBlockM));
  PBG_TRY(make_tmap(c, &st.tm_xd0, st.xd0, cap, c->kd0p, kBlockM));
  st.cap = cap;
  return PBG_OK;
}

int ensure_latents(pbg_ctx* c, long long rows, cudaStream_t stream) {
  if (c->lat_cap >= rows) return PBG_OK;
  PBG_TRY(begin_growth(c, stream, "the latent workspace"));
  const long long cap = pow2_cap(rows);
  c->lat_cap = 0;
  PBG_TRY(realloc_dev(c, c->lat_z, sizeof(float) * cap * c->dims.noise_dim));
  c->lat_cap = cap;
  return PBG_OK;
}

// torch splits a tensor of 2^31 elements or more into several launches, each with its own geometry and offset
int check_draw_size(pbg_ctx* c, long long total_rows) {
  if (total_rows < 1) return fail(c, PBG_ERR_INVALID, "latent draw: total_rows must be positive");
  if (total_rows > 0x7fffffffll / c->dims.noise_dim)
    return fail(c, PBG_ERR_UNSUPPORTED, "latent draw: %lld x %d elements is above the 2^31 - 1 of one torch launch",
                total_rows, c->dims.noise_dim);
  return PBG_OK;
}

// Rows [row_begin, row_begin + rows) of a [total_rows, Z] draw (latent.cuh) into out, at Philox (seed, offset) --
// or at (seed, st->offset) when st is given, advancing st->offset past the whole draw when `advance`.
int launch_draw(pbg_ctx* c, unsigned long long seed, unsigned long long offset, LatentStream* st, bool advance,
                long long total_rows, long long row_begin, long long rows, float* out, cudaStream_t s) {
  if (rows <= 0) return PBG_OK;
  const long long Z = c->dims.noise_dim;
  const LatentGeometry g = latent_geometry(total_rows * Z, c->num_sms, c->max_threads_sm);
  LatentParams p{};
  p.seed = seed; p.offset = offset; p.st = st; p.advance = advance ? 1 : 0; p.inc = g.inc; p.T = g.T;
  p.e_begin = row_begin * Z; p.e_end = (row_begin + rows) * Z; p.out = out;
  const long long r_lo = p.e_begin / (4 * g.T), r_hi = (p.e_end - 1) / (4 * g.T);
  p.slot_begin = r_lo * g.T;
  const long long blocks = (r_hi - r_lo + 1) * g.T / kLatentThreads;   // T is a multiple of the block
  { LaunchScope ls(c, PBG_K_OTHER, s);
    latent_draw_kernel<<<static_cast<unsigned>(blocks), kLatentThreads, 0, s>>>(p); }
  PBG_CUDA(c, cudaGetLastError());
  return PBG_OK;
}

// Draw a request's latents from the ctx's stream (staging: the whole request at once).
int draw_stream(pbg_ctx* c, long long B, float* out, cudaStream_t s) {
  PBG_TRY(check_draw_size(c, B));
  return launch_draw(c, c->lat_seed, 0, c->lat_st, true, B, 0, B, out, s);
}

template <int ACT>
int launch_f32(pbg_ctx* c, int kind, const Linear& l, const float* A, long long lda, float* out, long long ldo, long long M,
               cudaStream_t s) {
  F32GemmParams p{A, lda, l.w_f32, l.k, l.b_f32, out, ldo, (int)M, l.n, l.k, c->dims.leaky_slope};
  dim3 grid((l.n + 63) / 64, (unsigned)((M + 63) / 64));
  { LaunchScope ls(c, kind, s);
    gemm_f32_kernel<ACT><<<grid, 256, 0, s>>>(p); }
  PBG_CUDA(c, cudaGetLastError());
  return PBG_OK;
}


// CTAs per launch of the pass kernel: one per SM unless PBG_GRID asks for fewer (several streams sharing the GPU)
int pass_grid(const pbg_ctx* c) {
  static const int env = [] { const char* e = getenv("PBG_GRID"); return e ? atoi(e) : 0; }();
  const int want = c->launch_ctas > 0 ? c->launch_ctas : env;
  return (want > 0 && want < c->num_sms) ? std::max(2, want) : c->num_sms;
}

struct Pass;
int launch_pass2(pbg_ctx* c, Workspace& w, const Pass& a, const GatherParams& gp, long long off, long long rows,
                 void* gen_out, float* scores, bool external_gather, const StageSlot* slot = nullptr, bool gather_ahead = false);

struct Pass {
  const float* node_emb = nullptr; long long N = 0;
  const float* rel_emb = nullptr;  long long R = 0;
  const long long *heads = nullptr, *rels = nullptr, *tails = nullptr;
  long long hs = 1, rs = 1, ts = 1;
  const float *h = nullptr, *r = nullptr, *t = nullptr, *z = nullptr;
  bool draw_z = false;   // z == nullptr with the latent stream on: each chunk draws its rows of ONE draw over B
  void* gen_out = nullptr; int out_dtype = PBG_DT_F32;
  float *gen_scores = nullptr, *logits = nullptr, *probs = nullptr;
  bool run_g = false, run_d = false;
  long long B = 0; int prec = PBG_PREC_BF16; cudaStream_t stream = nullptr;
};

int run_chunk(pbg_ctx* c, const Pass& a, long long off, long long rows) {
  const int E = c->dims.embed_dim, Z = c->dims.noise_dim;
  const bool bf = a.prec == PBG_PREC_BF16;
  Workspace& w = bf ? c->ws_bf16 : c->ws_f32;
  cudaStream_t s = a.stream;

  GatherParams gp{};
  gp.node_emb = a.node_emb; gp.rel_emb = a.rel_emb; gp.N = a.N; gp.R = a.R; gp.E = E; gp.Z = Z;
  gp.heads = a.heads ? a.heads + off * a.hs : nullptr; gp.head_stride = a.hs;
  gp.rels = a.rels ? a.rels + off * a.rs : nullptr;    gp.rel_stride = a.rs;
  gp.tails = a.tails ? a.tails + off * a.ts : nullptr; gp.tail_stride = a.ts;
  gp.h = a.h ? a.h + off * E : nullptr; gp.r = a.r ? a.r + off * E : nullptr; gp.t = a.t ? a.t + off * E : nullptr;
  gp.z = a.z ? a.z + off * Z : nullptr;
  if (a.draw_z) {
    PBG_TRY(launch_draw(c, c->lat_seed, 0, c->lat_st, off + rows == a.B, a.B, off, rows, c->lat_z, s));
    gp.z = c->lat_z;
  }
  gp.xg = a.run_g ? w.xg0 : nullptr; gp.ldg = bf ? c->kg0p : c->kg0;
  gp.xd = a.run_d ? w.xd0 : nullptr; gp.ldd = bf ? c->kd0p : c->kd0;
  gp.B = rows; gp.err_flag = c->err_flag;
  const int gather_blocks = (int)std::min<long long>((rows + 7) / 8, (long long)c->num_sms * 8);
  if (!bf && (c->n_mirror > 0 || c->mc_gen || c->mc_cos || c->mc_logits || c->mc_probs))
    return fail(c, PBG_ERR_UNSUPPORTED, "result mirrors / multicast are a bf16-mode feature");
  // bf16 mode gathers inside the fused pass kernel.  PBG_SPLIT_GATHER=1 (experiment, see DESIGN.md 3.1 "time model"):
  // the rows are gathered by this small kernel instead -- it fits beside resident pass CTAs of other lanes (no shared
  // memory, few registers), so a pass no longer holds its SMs through a gather phase with idle tensor pipes.
  static const bool split_env = [] { const char* e = getenv("PBG_SPLIT_GATHER"); return e && atoi(e) != 0; }();
  const bool split = bf && split_env && rows > 0;
  if (!bf) {
    LaunchScope ls(c, PBG_K_GATHER, s);
    gather_concat_kernel<float><<<gather_blocks, 256, 0, s>>>(gp);
  } else if (split) {
    LaunchScope ls(c, PBG_K_GATHER, s);
    gather_concat_kernel<__nv_bfloat16><<<gather_blocks, 256, 0, s>>>(gp);
  }
  PBG_CUDA(c, cudaGetLastError());

  const size_t out_es = a.out_dtype == PBG_DT_BF16 ? 2 : 4;
  void* gen_out = a.gen_out ? static_cast<char*>(a.gen_out) + (size_t)off * E * out_es : nullptr;
  float* scores = a.gen_scores ? a.gen_scores + off : nullptr;

  if (bf) {
    return launch_pass2(c, w, a, gp, off, rows, gen_out, scores, split);
  } else {
    float *xg0 = (float*)w.xg0, *xd0 = (float*)w.xd0, *bufA = (float*)w.bufA, *bufB = (float*)w.bufB;
    const int row_blocks = (int)std::min<long long>((rows + 7) / 8, (long long)c->num_sms * 8);
    if (a.run_g) {
      const int H = c->dims.g_hidden;
      PBG_TRY(launch_f32<ACT_LEAKY>(c, PBG_K_G_L0, c->g[0], xg0, c->kg0, bufA, H, rows, s));
      PBG_TRY(launch_f32<ACT_LEAKY>(c, PBG_K_G_L1, c->g[1], bufA, H, bufB, H, rows, s));
      float* pred = gen_out ? (float*)gen_out : bufA;  // bufA is free once layer 2 has consumed it
      PBG_TRY(launch_f32<ACT_TANH>(c, PBG_K_G_L2, c->g[2], bufB, H, pred, E, rows, s));
      if (scores) {
        { LaunchScope ls(c, PBG_K_OTHER, s);
          cosine_f32_kernel<<<row_blocks, 256, 0, s>>>(pred, E, a.node_emb, a.N, a.tails + off * a.ts, a.ts, E, rows,
                                                       scores); }
        PBG_CUDA(c, cudaGetLastError());
      }
    }
    if (a.run_d) {
      const int H = c->dims.d_hidden, H2 = c->hd2;
      PBG_TRY(launch_f32<ACT_LEAKY>(c, PBG_K_D_L0, c->d[0], xd0, c->kd0, bufA, H, rows, s));
      PBG_TRY(launch_f32<ACT_LEAKY>(c, PBG_K_D_L1, c->d[1], bufA, H, bufB, H2, rows, s));
      { LaunchScope ls(c, PBG_K_OTHER, s);
        rowdot_f32_kernel<<<row_blocks, 256, 0, s>>>(bufB, H2, c->d_w3, c->d_b3, H2, rows, a.logits + off,
                                                     a.probs ? a.probs + off : nullptr); }
      PBG_CUDA(c, cudaGetLastError());
    }
  }
  return PBG_OK;
}


// launch with programmatic stream serialisation (pdl): the kernel may begin while its predecessor on the stream drains; it
// orders itself behind the predecessor with griddepcontrol.wait (topk_kernel.cuh: pdl_wait).  Used for the pass kernel
// (PBG_PDL) and, in top-k, for the kernels of one CTA per SM (sample, scan: their prologue -- barriers, TMEM,
// descriptors -- overlaps the predecessor's tail) and for the exact-scan launch.  NOT for the cut-off and rescoring kernels: their many small blocks, released early, pile onto
// whichever SMs the cluster kernel before them left idle (20 of 148 behind the sample launch, 34 behind a 1024-row scan)
// instead of spreading over the device -- measured per link at k = 64: cut-off +12 / +32 us at B = 1024 / 4096, rescore
// +33 us at B = 1024; sample, scan, exact: -3 us each (B = 256, k = 10: 84.5 -> 76 us).
template <class... KArgs, class... Args>
cudaError_t launch_pdl(bool pdl, void (*kern)(KArgs...), unsigned grid, unsigned block, size_t smem, cudaStream_t s, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(block); cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

// The pass kernel's instantiations, indexed by (TR ? 4 : 0) | (FASTG ? 2 : 0) | (BIASS ? 1 : 0).
using Pass2Kernel = void (*)(Pass2Params);
const Pass2Kernel kPass2[8] = {
    pbg_pass2_kernel<false, false, false>, pbg_pass2_kernel<false, false, true>, pbg_pass2_kernel<false, true, false>,
    pbg_pass2_kernel<false, true, true>,   pbg_pass2_kernel<true, false, false>, pbg_pass2_kernel<true, false, true>,
    pbg_pass2_kernel<true, true, false>,   pbg_pass2_kernel<true, true, true>};

// Per layer kind (IT_*): its epilogue, the counter that gates its A operand, the counter its stores bump.
const int kEpiOf[5] = {PEPI_STORE, PEPI_STORE, PEPI_STORE, PEPI_ROWDOT, PEPI_TANH};
const int kPredOf[5] = {DEP_X, DEP_X, DEP_G0, DEP_D0, DEP_G1};
const int kOutOf[5] = {DEP_G0, DEP_D0, DEP_G1, -1, -1};

// Layer kind k of a pass over Linear l: its A operand `amap`, the store map `omap` and rows `out` (leading dimension
// `ldo`) of a PEPI_STORE layer.  Tiles are 256 x 256, or 256 x 128 when the padded width is not a multiple of 256.
void set_layer(Pass2Params& p, int k, const Linear& l, const CUtensorMap& amap, const CUtensorMap* omap,
               __nv_bfloat16* out, int ldo) {
  const int bn = (l.np % 256 == 0) ? 256 : 128;
  p.tm_a[k] = amap;
  p.tm_w[k] = bn == 256 ? l.tmap_w128 : l.tmap_w64;
  if (omap) p.tm_o[k] = *omap;
  p.layer[k] = P2Layer{l.kp / kBlockK, bn, l.np / bn, kEpiOf[k], kPredOf[k], kOutOf[k], ldo, -1, l.b_pad, out};
  p.layer_mask |= 1u << k;
}

// The pair kernel (pass2_kernel.cuh): 256-row blocks, tiles of 256 x {256 | 128}, one CTA pair per tile.
int launch_pass2(pbg_ctx* c, Workspace& w, const Pass& a, const GatherParams& gp, long long off, long long rows,
                 void* gen_out, float* scores, bool external_gather, const StageSlot* slot, bool gather_ahead) {
  const int grid = pass_grid(c) & ~1;  // whole pairs
  Pass2Params p;
  memset(&p, 0, sizeof p);
  const Linear* lin[5] = {&c->g[0], &c->d[0], &c->g[1], &c->d[1], &c->g[2]};
  // first-layer operands: the ctx's own gather buffers, or a staged request's (pbg_stage_triplets)
  const CUtensorMap* amap[5] = {slot ? &slot->tm_xg0 : &w.tm_xg0, slot ? &slot->tm_xd0 : &w.tm_xd0, &w.tm_bufA_g, &w.tm_bufD_d,
                                &w.tm_bufB_g};
  const CUtensorMap* omap[5] = {&w.tmo_bufA, &w.tmo_bufD, &w.tmo_bufB, nullptr, nullptr};
  const bool on[5] = {a.run_g, a.run_d, a.run_g, a.run_d, a.run_g};
  const int nrb = static_cast<int>((rows + kP2Rows - 1) / kP2Rows);
  __nv_bfloat16* outs[5] = {(__nv_bfloat16*)w.bufA, (__nv_bfloat16*)w.bufD, (__nv_bfloat16*)w.bufB, nullptr, nullptr};
  const int ldos[5] = {c->hgp, c->hdp, c->hgp, 0, 0};
  long long total = 0;
  for (int k = 0; k < 5; ++k) {
    if (!on[k]) continue;
    set_layer(p, k, *lin[k], *amap[k], omap[k], outs[k], ldos[k]);
    if (p.layer[k].n_tiles > 255) return fail(c, PBG_ERR_UNSUPPORTED, "layer too wide for the tile index");
    total += static_cast<long long>(nrb) * p.layer[k].n_tiles;
  }
  // biases + final dot weights are copied to shared memory at kernel start when they fit (H <= 1024)
  bool biass = false;
  {
    int off = 0;
    for (int k = 0; k < 5; ++k) if (on[k]) { p.layer[k].bias_off = off; off += lin[k]->np; }
    p.w3_off = off;
    if (on[IT_D_L1]) off += lin[IT_D_L1]->np;
    biass = off <= P2Smem::kBiasFloats;
  }
  if (on[IT_D_L1] && lin[IT_D_L1]->np / 64 > kPartSlotsD) return fail(c, PBG_ERR_UNSUPPORTED, "d_hidden too wide for the partial buffer");
  if (on[IT_G_L2] && lin[IT_G_L2]->np / 64 > kPartSlotsG / 2) return fail(c, PBG_ERR_UNSUPPORTED, "embed_dim too wide for the partial buffer");
  // The gather ("phase 0"): every row of the pass in 4-row groups that the epilogue warps claim from a counter -- one
  // group each up front, the rest whenever a warp would otherwise wait (pass2_kernel.cuh).  Every tile is a static
  // ticket, layer by layer (a topological order); the scheduler thread polls a ticket's dependency counter.
  p.phase0_groups = external_gather ? 0 : nrb * kP2GroupsPerBlock;
  p.gather_external = external_gather ? 1 : 0;
  if (gather_ahead) {   // gp describes the NEXT request, gathered into the other staging slot while this pass runs
    p.phase0_groups = static_cast<int>((gp.B + 3) / 4);
    p.gather_ahead = 1;
  }
  {
    // Waves: the row blocks can be cut into `waves` groups whose layer phases are interleaved (L0 of every wave,
    // then L1 of every wave, then L2).  One wave measured best at every size (PBG_WAVES to experiment).
    static const int waves_env = [] { const char* e = getenv("PBG_WAVES"); return e ? atoi(e) : 1; }();
    const int waves = std::max(1, std::min(waves_env, std::min(nrb, 3)));
    // Ticket order (a topological order of the layer graph): L0 of both models, then L1 of both, then the generator's
    // L2.  PBG_MIX=1 instead interleaves, per row block, the discriminator's L1 tiles (MMA-bound) with the generator's
    // L2 tile (epilogue-bound: tanh, cosine, output rows); measured on B200 it changes nothing at 6 lanes x 48 SMs
    // (196.5 vs 197.0 M samples/s) or at B = 32768 (167.9 vs 167.1 us) and costs a single 48-SM pass 8 % -- off.
    static const int mix_env = [] { const char* e = getenv("PBG_MIX"); return e ? atoi(e) : 0; }();
    const bool mix = on[IT_D_L1] && on[IT_G_L2] && mix_env != 0;
    int start = 0;
    auto add_seg = [&](int k, int rb_lo, int rb_hi, int k2 = -1) {
      if (k < 0 || !on[k] || rb_hi == rb_lo) return;
      const int nt2 = (k2 >= 0 && on[k2]) ? p.layer[k2].n_tiles : 0;
      p.seg[p.n_seg++] = P2Segment{k, p.layer[k].n_tiles, start, rb_lo, nt2 ? k2 : k, nt2};
      start += (rb_hi - rb_lo) * (p.layer[k].n_tiles + nt2);
    };
    for (int wv = 0; wv < waves; ++wv) {
      const int rb_lo = static_cast<int>(static_cast<long long>(nrb) * wv / waves);
      const int rb_hi = static_cast<int>(static_cast<long long>(nrb) * (wv + 1) / waves);
      add_seg(IT_G_L0, rb_lo, rb_hi);
      add_seg(IT_D_L0, rb_lo, rb_hi);
    }
    add_seg(IT_G_L1, 0, nrb);
    if (mix) {
      add_seg(IT_D_L1, 0, nrb, IT_G_L2);
    } else {
      add_seg(IT_D_L1, 0, nrb);
      add_seg(IT_G_L2, 0, nrb);
    }
    if (start != total) return fail(c, PBG_ERR_INVALID, "internal: static item list does not cover the pass");
    p.n_total = start;
  }
  p.gather = gp;
  static const int poll_env = [] { const char* e = getenv("PBG_POLL_NS"); return e ? atoi(e) : 40; }();
  p.poll_ns = poll_env;
  static const int defer_env = [] { const char* e = getenv("PBG_GATHER_DEFER"); return e ? atoi(e) : 1; }();
  p.gather_defer = defer_env;
  // dead workspace row blocks are dropped from L2 instead of being written back to HBM (pass2_kernel.cuh: p2_discard;
  // in rotation over six lanes' workspaces: 31.9 -> 1.9 MB of DRAM writes per 4096-triplet launch,
  // profiles/dram_steady_r2.txt)
  p.discard = c->discard;
  // the first-layer operand rows are this pass's to drop when it gathered them itself into the ctx's own buffers, or when
  // it consumes a staging slot (pbg_score_staged_stage_next); a slot scored by pbg_score_staged may be scored again
  if (!external_gather) {
    p.dead_xg = gp.xg; p.dead_xd = gp.xd;
  } else if (gather_ahead && slot) {
    p.dead_xg = a.run_g ? slot->xg0 : nullptr; p.dead_xd = a.run_d ? slot->xd0 : nullptr;
  }
  p.dead_ldg = c->kg0p; p.dead_ldd = c->kd0p;
  p.nrb = nrb; p.rb_cap = w.mb_cap; p.M = static_cast<int>(rows); p.slope = c->dims.leaky_slope;
  p.sched = w.sched; p.ready = w.ready; p.fin = w.fin;
  p.gen_out = gen_out; p.out_f32 = a.out_dtype == PBG_DT_F32; p.n_valid = c->dims.embed_dim; p.ld_gen = c->dims.embed_dim;
  if (scores && slot && slot->has_xt) {   // the staging kernel left the tail rows, in request order, in the slot
    p.cosine = scores; p.tail_tab = slot->xt; p.n_ent = slot->cap; p.tail_idx = nullptr; p.tail_stride = 0;
  } else if (scores && slot) {             // staged by the previous pass: the tail rows are read through the request's ids
    p.cosine = scores; p.tail_tab = slot->node_emb; p.n_ent = slot->N; p.tail_idx = slot->tails; p.tail_stride = 3;
  } else if (scores) {
    p.cosine = scores; p.tail_tab = a.node_emb; p.n_ent = a.N;
    p.tail_idx = a.tails + off * a.ts; p.tail_stride = a.ts;
  }
  p.part_g = w.part_g; p.slots_g = on[IT_G_L2] ? (c->dims.embed_dim + 63) / 64 : 0;  // only the valid columns
  p.w3 = c->d_w3_pad; p.b3 = c->d_b3;
  p.logits = a.logits ? a.logits + off : nullptr;
  p.probs = a.probs ? a.probs + off : nullptr;
  p.part_d = w.part_d; p.slots_d = on[IT_D_L1] ? lin[IT_D_L1]->np / 64 : 0;
  p.trace = c->trace;
  p.n_mirror = c->n_mirror;
  for (int i = 0; i < c->n_mirror; ++i) {
    if (gen_out && !c->mir_gen[i]) return fail(c, PBG_ERR_INVALID, "result mirror %d has no gen_out buffer", i);
    if (scores && !c->mir_cos[i]) return fail(c, PBG_ERR_INVALID, "result mirror %d has no gen_scores buffer", i);
    if (a.logits && !c->mir_logits[i]) return fail(c, PBG_ERR_INVALID, "result mirror %d has no logits buffer", i);
    const size_t es = a.out_dtype == PBG_DT_BF16 ? 2 : 4;
    p.mir_gen[i] = c->mir_gen[i] ? static_cast<char*>(c->mir_gen[i]) + static_cast<size_t>(off) * c->dims.embed_dim * es : nullptr;
    p.mir_cos[i] = c->mir_cos[i] ? c->mir_cos[i] + off : nullptr;
    p.mir_logits[i] = c->mir_logits[i] ? c->mir_logits[i] + off : nullptr;
    p.mir_probs[i] = (c->mir_probs[i] && a.probs) ? c->mir_probs[i] + off : nullptr;
  }
  {
    const size_t es = a.out_dtype == PBG_DT_BF16 ? 2 : 4;
    p.mc_gen = (c->mc_gen && gen_out) ? static_cast<char*>(c->mc_gen) + static_cast<size_t>(off) * c->dims.embed_dim * es : nullptr;
    p.mc_cos = (c->mc_cos && scores) ? c->mc_cos + off : nullptr;
    p.mc_logits = (c->mc_logits && a.logits) ? c->mc_logits + off : nullptr;
    p.mc_probs = (c->mc_probs && a.probs) ? c->mc_probs + off : nullptr;
  }
  // programmatic dependent launch: this pass may begin its prologue while the previous kernel of the stream drains
  static const bool pdl = [] { const char* e = getenv("PBG_PDL"); return !e || atoi(e) != 0; }();
  const bool fastg = c->dims.embed_dim == 128 && c->dims.noise_dim % 4 == 0 && c->dims.noise_dim <= 128 &&
                     c->kg0p == c->kg0 && c->kd0p == c->kd0;  // the bulk-store gather writes unpadded rows
  const Pass2Kernel kern = kPass2[(p.trace ? 4 : 0) | (fastg ? 2 : 0) | (biass ? 1 : 0)];
  cudaError_t le;
  { LaunchScope ls(c, PBG_K_PASS, a.stream);
    le = launch_pdl(pdl, kern, grid, kP2Threads, P2Smem::kTotal, a.stream, p); }
  if (le == cudaSuccess) le = cudaGetLastError();
  if (le != cudaSuccess) {
    cudaFuncAttributes fa{};
    cudaFuncGetAttributes(&fa, kern);
    return fail(c, PBG_ERR_CUDA, "pass kernel launch failed: %s (grid %d x %d threads, %d regs/thread, %zu B static + %d B dynamic smem, "
                "max threads/block %d, max dynamic smem %d)", cudaGetErrorString(le), grid, kP2Threads, fa.numRegs,
                fa.sharedSizeBytes, P2Smem::kTotal, fa.maxThreadsPerBlock, fa.maxDynamicSharedSizeBytes);
  }
  return PBG_OK;
}

int run_pass(pbg_ctx* c, Pass a) {
  if (!c) return PBG_ERR_INVALID;
  if (a.B < 0) return fail(c, PBG_ERR_INVALID, "negative batch");
  if (a.prec != PBG_PREC_F32 && a.prec != PBG_PREC_BF16) return fail(c, PBG_ERR_INVALID, "unknown precision %d", a.prec);
  if (a.run_g && !c->g_loaded) return fail(c, PBG_ERR_NOT_LOADED, "generator weights not loaded");
  if (a.run_d && !c->d_loaded) return fail(c, PBG_ERR_NOT_LOADED, "discriminator weights not loaded");
  if (a.run_g && a.z == nullptr && !c->lat_on) return fail(c, PBG_ERR_INVALID, "generator needs latents z");
  a.draw_z = a.run_g && a.z == nullptr && a.B > 0;
  if (a.draw_z) PBG_TRY(check_draw_size(c, a.B));
  if (a.run_g && a.gen_out && a.prec == PBG_PREC_F32 && a.out_dtype != PBG_DT_F32)
    return fail(c, PBG_ERR_INVALID, "fp32 mode writes fp32 output");
  if (a.gen_scores && a.tails == nullptr) return fail(c, PBG_ERR_INVALID, "gen_scores needs tail ids");
  if (a.B == 0 || (!a.run_g && !a.run_d)) return PBG_OK;
  PBG_CUDA(c, cudaSetDevice(c->dims.device));
  const long long chunk = std::min(a.B, kMaxChunk);
  PBG_TRY(ensure_ws(c, a.prec, chunk, a.stream));
  if (a.draw_z) PBG_TRY(ensure_latents(c, chunk, a.stream));
  for (long long off = 0; off < a.B; off += chunk) PBG_TRY(run_chunk(c, a, off, std::min(chunk, a.B - off)));
  return PBG_OK;
}

}  // namespace

extern "C" {

int pbg_abi_version(void) { return PBG_ABI_VERSION; }

const char* pbg_last_error(const pbg_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int64_t pbg_launch_count(const pbg_ctx* ctx) { return ctx ? ctx->launches : 0; }

int64_t pbg_format_f32_json(const float* v, size_t rows, int cols, int indent, int depth, char* out, size_t cap) {
  if ((!v && rows) || cols < 0 || depth < 0) return -(int64_t)fail(nullptr, PBG_ERR_INVALID, "format_f32_json: bad arguments");
  return (int64_t)pbg_host::format_rows<float>(v, rows, cols, indent, depth, out, cap, pbg_host::put_py_float);
}

int64_t pbg_format_i64_json(const int64_t* v, size_t rows, int cols, int indent, int depth, char* out, size_t cap) {
  if ((!v && rows) || cols < 0 || depth < 0) return -(int64_t)fail(nullptr, PBG_ERR_INVALID, "format_i64_json: bad arguments");
  return (int64_t)pbg_host::format_rows<int64_t>(v, rows, cols, indent, depth, out, cap, pbg_host::put_i64);
}

int64_t pbg_parse_index_rows(const char* text, size_t len, int cols, int64_t* out, size_t cap_rows) {
  if (!text || cols < 1 || cols > 8) return -(int64_t)fail(nullptr, PBG_ERR_INVALID, "parse_index_rows: null text or cols outside 1..8");
  const char* msg = nullptr;
  size_t off = 0;
  const long long rows = pbg_host::parse_index_rows(text, len, cols, out, cap_rows, &msg, &off);
  if (rows < 0) return -(int64_t)fail(nullptr, PBG_ERR_INVALID, "parse_index_rows: %s at byte %zu", msg, off);
  return rows;
}

int pbg_topk_prepare(pbg_ctx* c, const float* table, int64_t N, void* stream) {
  if (!c) return PBG_ERR_INVALID;
  if (!table || N <= 0) return fail(c, PBG_ERR_INVALID, "topk: null or empty table");
  const int E = c->dims.embed_dim;
  if (E % 4) return fail(c, PBG_ERR_UNSUPPORTED, "topk: embed_dim must be a multiple of 4");
  PBG_CUDA(c, cudaSetDevice(c->dims.device));
  cudaStream_t s = (cudaStream_t)stream;
  TopkState& t = c->tk;
  const long long n_pad = (N + 255) / 256 * 256;
  if (n_pad != t.n_pad) {
    PBG_TRY(begin_growth(c, s, "the top-k table"));
    t.n_pad = 0;
    PBG_TRY(realloc_dev(c, t.tn, sizeof(__nv_bfloat16) * n_pad * E));
    PBG_TRY(realloc_dev(c, t.inv_t, sizeof(float) * n_pad));
    t.n_pad = n_pad;
    if (E == 128) PBG_TRY(make_tmap(c, &t.tm_t, t.tn, n_pad, E, 128));
  }
  t.table = table; t.N = N;
  { LaunchScope ls(c, PBG_K_OTHER, s);
    if (E <= 128) topk_prepare_kernel<8, 1><<<c->num_sms * 8, 256, 0, s>>>(table, N, n_pad, E, t.tn, t.inv_t);
    else topk_prepare_kernel<2, 4><<<c->num_sms * 8, 256, 0, s>>>(table, N, n_pad, E, t.tn, t.inv_t); }
  PBG_CUDA(c, cudaGetLastError());
  return PBG_OK;
}

// Largest k the general path serves: the selection kernel keeps k (score, index) pairs per thread in shared memory.
constexpr int kTkGeneralMaxK = 512;

namespace {
// General path (k > kTkMaxK, E != 128, small tables): exact fp32 scores of a chunk of rows through the SIMT GEMM of the
// parity mode (raw dot products; the row norms are applied by the selection kernel), then one selection CTA per row.
int topk_general(pbg_ctx* c, TopkState& t, const float* q, long long rows, int k, long long* oi, float* os, cudaStream_t s) {
  const int E = c->dims.embed_dim;
  const long long chunk = std::max<long long>(64, std::min<long long>(rows, (512ll << 20) / (4 * t.N)));
  const size_t need = static_cast<size_t>(chunk) * t.N;
  if (t.score_cap < need) {
    PBG_TRY(begin_growth(c, s, "the top-k score buffer"));
    t.score_cap = 0;
    PBG_TRY(realloc_dev(c, t.score_buf, sizeof(float) * need));
    t.score_cap = need;
  }
  const int threads = std::max(32, std::min(256, (200 * 1024 / (k * 8)) / 32 * 32));
  const size_t smem = static_cast<size_t>(E) * 4 + static_cast<size_t>(threads) * k * 8;
  for (long long off = 0; off < rows; off += chunk) {
    const long long r = std::min(chunk, rows - off);
    F32GemmParams gp{q + off * E, E, t.table, E, nullptr, t.score_buf, t.N, (int)r, (int)t.N, E, 0.f};
    dim3 grid((unsigned)((t.N + 63) / 64), (unsigned)((r + 63) / 64));
    { LaunchScope ls(c, PBG_K_OTHER, s);
      gemm_f32_kernel<ACT_NONE><<<grid, 256, 0, s>>>(gp); }
    PBG_CUDA(c, cudaGetLastError());
    // selection: histogram + sort per row (topk_select_kernel); a row it cannot take (thousands of equal scores at the
    // cut) is flagged and redone by the per-thread-list kernel
    { LaunchScope ls(c, PBG_K_OTHER, s);
      topk_select_kernel<<<static_cast<unsigned>(std::min<long long>(r, 6ll * c->num_sms)), kSelThreads, 0, s>>>(
          t.score_buf, t.inv_q + off, t.inv_t, t.N, k, r, oi + off * k, os + off * k, t.flag + off); }
    PBG_CUDA(c, cudaGetLastError());
    { LaunchScope ls(c, PBG_K_OTHER, s);
      topk_exact_kernel<<<static_cast<unsigned>(std::min<long long>(r, 2ll * c->num_sms)), threads, smem, s>>>(
          q + off * E, t.inv_q + off, t.table, t.inv_t, t.N, E, k, t.flag + off, 0, t.score_buf, oi + off * k, os + off * k, r); }
    PBG_CUDA(c, cudaGetLastError());
  }
  return PBG_OK;
}
}  // namespace

int pbg_topk(pbg_ctx* c, const float* queries, int64_t B, int k, int64_t* out_idx, float* out_scores, void* stream) {
  if (!c) return PBG_ERR_INVALID;
  TopkState& t = c->tk;
  if (B < 0) return fail(c, PBG_ERR_INVALID, "negative batch");
  if (B == 0) return PBG_OK;
  if (!t.table) return fail(c, PBG_ERR_NOT_LOADED, "topk: no table prepared (pbg_topk_prepare)");
  if (!queries || !out_idx || !out_scores) return fail(c, PBG_ERR_INVALID, "null tensor");
  if (k < 1) return fail(c, PBG_ERR_INVALID, "topk: k must be positive");
  if (k > t.N) return fail(c, PBG_ERR_INVALID, "topk: k = %d exceeds the %lld rows of the table", k, t.N);  // torch raises too
  if (k > kTkGeneralMaxK) return fail(c, PBG_ERR_UNSUPPORTED, "topk: k = %d is above the %d this library selects on the device", k, kTkGeneralMaxK);
  PBG_CUDA(c, cudaSetDevice(c->dims.device));
  cudaStream_t s = (cudaStream_t)stream;
  const int E = c->dims.embed_dim;
  // rows per round of launches.  A row's cut-off is the k-th best of its sampled group keys, 16 kept per (row, pair, column
  // half) list: at 4096 rows a block is met by 5-6 pairs in the sample launch (160+ keys), at 16384 rows by 2-3 -- enough
  // for k <= 16 only
  const long long kChunk = k > 16 ? 4096 : 16384;
  // small tables / other shapes: the general path.  The sample launch sees N / (32 stride) groups of 32 entities per row
  // and the cut-off needs k positive group maxima among them: at least 2 k groups
  // The cut-off is the k-th best score of a 1-in-`stride` sample of the table tiles, so about stride * k entities (+ a dozen
  // inside the error margin) pass it and are rescored: the stride shrinks as k grows (k = 64 at 1 in 8: one row in a
  // hundred had more than the 1024 candidates the rescoring kernel takes and went to the 3 ms exact scan).
  const int stride = tk_sample_stride(k);
  const bool filter = E == 128 && k <= kTkMaxK && t.N >= std::max<long long>(16 * 256, 64ll * stride * k);
  for (long long off = 0; off < B; off += kChunk) {
    const long long rows = std::min(kChunk, B - off);
    const long long rows_pad = (rows + 255) / 256 * 256;
    const float* q = queries + off * E;
    if (t.q_cap < rows_pad) {
      PBG_TRY(begin_growth(c, s, "the top-k query buffers"));
      t.q_cap = 0;
      PBG_TRY(realloc_dev(c, t.qn, sizeof(__nv_bfloat16) * rows_pad * E));
      PBG_TRY(realloc_dev(c, t.inv_q, sizeof(float) * rows_pad));
      PBG_TRY(realloc_dev(c, t.flag, sizeof(int) * rows_pad));
      PBG_TRY(realloc_dev(c, t.tau, sizeof(float) * rows_pad));
      t.q_cap = rows_pad;
      if (E == 128) PBG_TRY(make_tmap(c, &t.tm_q, t.qn, rows_pad, E, 128));
    }
    { LaunchScope ls(c, PBG_K_OTHER, s);
      const unsigned pg = static_cast<unsigned>(std::min<long long>(c->num_sms * 8, (rows_pad + 7) / 8));
      if (E <= 128) topk_prepare_kernel<8, 1><<<pg, 256, 0, s>>>(q, rows, rows_pad, E, t.qn, t.inv_q);
      else topk_prepare_kernel<2, 4><<<pg, 256, 0, s>>>(q, rows, rows_pad, E, t.qn, t.inv_q); }
    PBG_CUDA(c, cudaGetLastError());
    long long* oi = reinterpret_cast<long long*>(out_idx) + off * k;
    float* os = out_scores + off * k;
    t.last_rows = rows; t.last_filtered = filter;
    if (!filter) {
      PBG_TRY(topk_general(c, t, q, rows, k, oi, os, s));
      continue;
    }
    const int grid = pass_grid(c) & ~1;
    const int npairs = grid / 2;
    const int n_rb = static_cast<int>(rows_pad / 256);
    const int n_tiles = static_cast<int>(t.n_pad / 256);
    // work units = query block x visited tile, query-block major; every pair takes an equal, contiguous span of them
    // (cut at query-block boundaries inside the kernel), so all SMs scan the same number of tiles whatever B is.  A
    // query block met by s pairs needs s list slots per row: the span is at least tiles / (kTkMaxRanges - 1).
    auto split = [&](int tiles, TopkParams& p, bool align) {
      p.n_rb = n_rb;
      p.n_tiles = tiles;
      p.total = n_rb * tiles;
      p.span = std::max({1, (p.total + npairs - 1) / npairs, (tiles + kTkMaxRanges - 2) / (kTkMaxRanges - 1)});
      // A span that crosses a query-block boundary costs its pair a second segment (new query tile, lists closed and
      // reopened: ~5 us).  The scan launch (56 tiles per pair at B = 4096) gains more from all 74 pairs being busy than
      // it loses (61 against 66 us); the sample launch (7 tiles per pair) does not (24 against 17 us), so its span is
      // rounded up to divide a query block's tiles: one segment per pair, fewer pairs.
      if (align && p.span < tiles) { const int pieces = std::max(1, tiles / p.span); p.span = (tiles + pieces - 1) / pieces; }
      p.n_ranges = 1;
      for (int rb = 0; rb < n_rb; ++rb)
        p.n_ranges = std::max(p.n_ranges, ((rb + 1) * tiles - 1) / p.span - (rb * tiles) / p.span + 1);
    };
    TopkParams ps, pm;
    memset(&ps, 0, sizeof ps); memset(&pm, 0, sizeof pm);
    ps.tm_q = pm.tm_q = t.tm_q; ps.tm_t = pm.tm_t = t.tm_t; ps.N = pm.N = t.N;
    ps.tile_stride = stride; pm.tile_stride = 1;
    split((n_tiles + stride - 1) / stride, ps, true);
    split(n_tiles, pm, false);
    const int n_slists = ps.n_ranges * 2, n_lists = pm.n_ranges * 2;
    const size_t need = static_cast<size_t>(rows_pad) * n_lists * kTkCand;
    const size_t sneed = static_cast<size_t>(rows_pad) * n_slists * kTkKeys;
    if (t.cand_cap < need || t.samp_cap < sneed) {
      PBG_TRY(begin_growth(c, s, "the top-k candidate buffers"));
      t.cand_cap = t.samp_cap = 0;
      PBG_TRY(realloc_dev(c, t.cand_grp, sizeof(unsigned) * need));
      PBG_TRY(realloc_dev(c, t.cand_mask, sizeof(unsigned) * need));
      PBG_TRY(realloc_dev(c, t.cand_cnt, sizeof(int) * need / kTkCand));
      PBG_TRY(realloc_dev(c, t.samp_keys, sizeof(int) * sneed));
      t.cand_cap = need; t.samp_cap = sneed;
    }
    ps.samp_keys = t.samp_keys;
    pm.tau = t.tau; pm.cand_grp = t.cand_grp; pm.cand_mask = t.cand_mask; pm.cand_cnt = t.cand_cnt;
    { LaunchScope ls(c, PBG_K_TOPK, s);
      PBG_CUDA(c, launch_pdl(true, pbg_topk_scan_kernel<TK_SAMPLE>, std::min(grid, 2 * ((ps.total + ps.span - 1) / ps.span)), kPassThreads, TkSmem::kTotal, s, ps)); }
    { LaunchScope ls(c, PBG_K_OTHER, s);
      PBG_CUDA(c, launch_pdl(false, topk_tau_kernel, static_cast<unsigned>((rows_pad + 7) / 8), 256, 0, s, t.samp_keys, n_slists, rows, rows_pad, k, t.tau)); }
    { LaunchScope ls(c, PBG_K_TOPK, s);
      PBG_CUDA(c, launch_pdl(true, pbg_topk_scan_kernel<TK_SCAN>, std::min(grid, 2 * ((pm.total + pm.span - 1) / pm.span)), kPassThreads, TkSmem::kTotal, s, pm)); }
    { LaunchScope ls(c, PBG_K_OTHER, s);
      PBG_CUDA(c, launch_pdl(false, topk_rescore_kernel, static_cast<unsigned>((rows + kTkRescoreWarps - 1) / kTkRescoreWarps), 32 * kTkRescoreWarps, 0, s,
                             q, t.inv_q, t.table, t.inv_t, t.cand_grp, t.cand_mask, t.cand_cnt, t.tau, n_lists, rows, t.N, k, oi, os, t.flag)); }
    { // rows the filter could not prove: exact scan, one CTA per row (rare)
      LaunchScope ls(c, PBG_K_OTHER, s);
      PBG_CUDA(c, launch_pdl(true, topk_exact_kernel, static_cast<unsigned>(std::min<long long>(rows, 2ll * c->num_sms)), 256,
                             static_cast<size_t>(E * 4 + 256 * k * 8), s, q, t.inv_q, t.table, t.inv_t, t.N, E, k, t.flag, 0, nullptr, oi, os, rows)); }
  }
  return PBG_OK;
}

int64_t pbg_topk_last_flagged(pbg_ctx* c, void* stream) {
  if (!c) return -1;
  TopkState& t = c->tk;
  if (!t.last_filtered || t.last_rows <= 0) return 0;
  if (cudaSetDevice(c->dims.device) != cudaSuccess) return -1;
  std::vector<int> h(static_cast<size_t>(t.last_rows));
  if (cudaMemcpyAsync(h.data(), t.flag, sizeof(int) * h.size(), cudaMemcpyDeviceToHost, (cudaStream_t)stream) != cudaSuccess) return -1;
  if (cudaStreamSynchronize((cudaStream_t)stream) != cudaSuccess) return -1;
  int64_t n = 0, why[5] = {0, 0, 0, 0, 0};
  for (int v : h) { n += v != 0; why[(v >= 0 && v <= 4) ? v : 0] += 1; }
  char buf[160];
  snprintf(buf, sizeof buf, "topk: %lld of %lld rows to the exact scan (list overflow %lld, too many candidates %lld, too few %lld, proof failed %lld)",
           (long long)n, t.last_rows, (long long)why[1], (long long)why[2], (long long)why[3], (long long)why[4]);
  c->err = buf;   // diagnostics text, readable through pbg_last_error
  return n;
}

int pbg_set_result_mirrors(pbg_ctx* c, int n, void* const* gen_out, float* const* gen_scores, float* const* logits,
                           float* const* probs) {
  if (!c) return PBG_ERR_INVALID;
  if (n < 0 || n > kMaxMirrors) return fail(c, PBG_ERR_INVALID, "at most %d result mirrors", kMaxMirrors);
  c->n_mirror = n;
  for (int i = 0; i < kMaxMirrors; ++i) {
    c->mir_gen[i] = (i < n && gen_out) ? gen_out[i] : nullptr;
    c->mir_cos[i] = (i < n && gen_scores) ? gen_scores[i] : nullptr;
    c->mir_logits[i] = (i < n && logits) ? logits[i] : nullptr;
    c->mir_probs[i] = (i < n && probs) ? probs[i] : nullptr;
  }
  return PBG_OK;
}

int pbg_set_result_multicast(pbg_ctx* c, void* gen_out_mc, float* gen_scores_mc, float* logits_mc, float* probs_mc) {
  if (!c) return PBG_ERR_INVALID;
  c->mc_gen = gen_out_mc; c->mc_cos = gen_scores_mc; c->mc_logits = logits_mc; c->mc_probs = probs_mc;
  return PBG_OK;
}

int pbg_set_launch_width(pbg_ctx* c, int n_ctas) {
  if (!c) return PBG_ERR_INVALID;
  if (n_ctas < 0) return fail(c, PBG_ERR_INVALID, "launch width must be >= 0");
  c->launch_ctas = n_ctas;
  return PBG_OK;
}

int pbg_last_pass_sm_clock(pbg_ctx* c, void* stream, double* mhz_out) {
  if (!c || !mhz_out) return PBG_ERR_INVALID;
  *mhz_out = 0.0;
  Workspace& w = c->ws_bf16;
  if (!w.sched) return fail(c, PBG_ERR_INVALID, "no bf16-mode pass has run on this ctx");
  PBG_CUDA(c, cudaSetDevice(c->dims.device));
  cudaStream_t s = (cudaStream_t)stream;
  PassSched h;
  PBG_CUDA(c, cudaMemcpyAsync(&h, w.sched, sizeof h, cudaMemcpyDeviceToHost, s));
  PBG_CUDA(c, cudaStreamSynchronize(s));
  if (h.clk_ns > 0) *mhz_out = static_cast<double>(h.clk_ticks) / static_cast<double>(h.clk_ns) * 1e3;
  return PBG_OK;
}

int pbg_set_workspace_discard(pbg_ctx* c, int on) {
  if (!c) return PBG_ERR_INVALID;
  c->discard = on ? 1 : 0;
  return PBG_OK;
}

int pbg_create(pbg_ctx** out, const pbg_dims* dims) {
  if (!out || !dims) return fail(nullptr, PBG_ERR_INVALID, "null argument");
  *out = nullptr;
  const int E = dims->embed_dim, Z = dims->noise_dim, HG = dims->g_hidden, HD = dims->d_hidden;
  if (E <= 0 || Z <= 0 || HG <= 0 || HD <= 0) return fail(nullptr, PBG_ERR_INVALID, "dims must be positive");
  if (!(dims->leaky_slope >= 0.f && dims->leaky_slope <= 1.f))
    return fail(nullptr, PBG_ERR_UNSUPPORTED, "leaky_slope must be in [0, 1]");
  if (E % 8 || Z % 8 || HG % 8 || HD % 16)
    return fail(nullptr, PBG_ERR_UNSUPPORTED, "embed_dim, noise_dim, g_hidden must be multiples of 8 and d_hidden of 16");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(nullptr, PBG_ERR_UNSUPPORTED, "no CUDA device (%s); this library has no CPU fallback",
                e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
  if (dims->device < 0 || dims->device >= ndev) return fail(nullptr, PBG_ERR_INVALID, "device %d out of range", dims->device);
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, dims->device)) != cudaSuccess)
    return fail(nullptr, PBG_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
  if (prop.major != 10)
    return fail(nullptr, PBG_ERR_UNSUPPORTED, "device %d is sm_%d%d; the kernels are sm_100a only (no fallback)",
                dims->device, prop.major, prop.minor);
  pbg_ctx* c = new (std::nothrow) pbg_ctx();
  if (!c) return fail(nullptr, PBG_ERR_NOMEM, "out of host memory");
  c->dims = *dims;
  c->num_sms = prop.multiProcessorCount;
  c->max_threads_sm = prop.maxThreadsPerMultiProcessor;
  if (const char* e = getenv("PBG_DISCARD")) c->discard = atoi(e) != 0;
  if (const char* e = getenv("PBG_HOST_SYNC")) c->host_block = strcmp(e, "block") == 0;
  c->kg0 = 2 * E + Z; c->kg0p = round_up(c->kg0, kBlockK);
  c->kd0 = 3 * E;     c->kd0p = round_up(c->kd0, kBlockK);
  c->hgp = round_up(HG, 128); c->hdp = round_up(HD, 128);
  c->hd2 = HD / 2;
  c->hmax = std::max(c->hgp, c->hdp);
  auto bail = [&](int code) { g_create_error = c->err; pbg_destroy(c); return code; };
  if (cudaSetDevice(dims->device) != cudaSuccess) { c->err = "cudaSetDevice failed"; return bail(PBG_ERR_CUDA); }
  // the dynamic shared memory of the kernels that take more than the default 48 KB, on this ctx's device
  e = cudaSuccess;
  for (Pass2Kernel k : kPass2)
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, P2Smem::kTotal);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(pbg_topk_scan_kernel<TK_SAMPLE>, cudaFuncAttributeMaxDynamicSharedMemorySize, TkSmem::kTotal);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(pbg_topk_scan_kernel<TK_SCAN>, cudaFuncAttributeMaxDynamicSharedMemorySize, TkSmem::kTotal);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(topk_exact_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024);
  if (e != cudaSuccess) { c->err = std::string("cudaFuncSetAttribute failed: ") + cudaGetErrorString(e); return bail(PBG_ERR_CUDA); }
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn) {
    c->err = "cuTensorMapEncodeTiled not available from the driver";
    return bail(PBG_ERR_CUDA);
  }
  c->encode = reinterpret_cast<EncodeTiledFn>(fn);
  if (cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaMalloc(&c->err_flag, sizeof(int)) != cudaSuccess ||
      cudaMemset(c->err_flag, 0, sizeof(int)) != cudaSuccess ||
      cudaMallocHost(&c->err_flag_host, sizeof(int)) != cudaSuccess ||
      cudaMalloc(&c->lat_st, sizeof(LatentStream)) != cudaSuccess ||
      cudaMemset(c->lat_st, 0, sizeof(LatentStream)) != cudaSuccess) {
    c->err = std::string("ctx allocation failed: ") + cudaGetErrorString(cudaGetLastError());
    return bail(PBG_ERR_CUDA);
  }
  *c->err_flag_host = 0;
  *out = c;
  return PBG_OK;
}

void pbg_destroy(pbg_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->dims.device);
  cudaDeviceSynchronize();
  for (auto& l : c->g) free_linear(l);
  for (auto& l : c->d) free_linear(l);
  cudaFree(c->d_w3); cudaFree(c->d_w3_pad);
  free_ws(c->ws_bf16); free_ws(c->ws_f32);
  free_stage(c->stage[0]); free_stage(c->stage[1]);
  cudaFree(c->err_flag); cudaFree(c->trace);
  cudaFree(c->lat_st); cudaFree(c->lat_z);
  cudaFree(c->tk.tn); cudaFree(c->tk.inv_t); cudaFree(c->tk.qn); cudaFree(c->tk.inv_q);
  cudaFree(c->tk.cand_grp); cudaFree(c->tk.cand_mask); cudaFree(c->tk.cand_cnt); cudaFree(c->tk.flag);
  cudaFree(c->tk.samp_keys); cudaFree(c->tk.tau); cudaFree(c->tk.score_buf);

  if (c->err_flag_host) cudaFreeHost(c->err_flag_host);
  if (c->host_evt) cudaEventDestroy(c->host_evt);
  cudaFree(c->st_block);
  if (c->own_stream) cudaStreamDestroy(c->own_stream);
  delete c;
}

int pbg_load_generator(pbg_ctx* c, const float* p, size_t n_floats) {
  if (!c || !p) return PBG_ERR_INVALID;
  const size_t E = c->dims.embed_dim, H = c->dims.g_hidden, K0 = c->kg0;
  const size_t want = H * K0 + H + H * H + H + E * H + E;
  if (n_floats != want) return fail(c, PBG_ERR_INVALID, "generator blob has %zu floats, expected %zu", n_floats, want);
  PBG_CUDA(c, cudaSetDevice(c->dims.device));
  c->g_loaded = false;
  const float* w1 = p;            const float* b1 = w1 + H * K0;
  const float* w2 = b1 + H;       const float* b2 = w2 + H * H;
  const float* w3 = b2 + H;       const float* b3 = w3 + E * H;
  PBG_TRY(upload_linear(c, c->g[0], (int)H, (int)K0, c->kg0p, w1, b1));
  PBG_TRY(upload_linear(c, c->g[1], (int)H, (int)H, c->hgp, w2, b2));
  PBG_TRY(upload_linear(c, c->g[2], (int)E, (int)H, c->hgp, w3, b3));
  c->g_loaded = true;
  return PBG_OK;
}

int pbg_load_discriminator(pbg_ctx* c, const float* p, size_t n_floats) {
  if (!c || !p) return PBG_ERR_INVALID;
  const size_t H = c->dims.d_hidden, H2 = c->hd2, K0 = c->kd0;
  const size_t want = H * K0 + H + H2 * H + H2 + H2 + 1;
  if (n_floats != want) return fail(c, PBG_ERR_INVALID, "discriminator blob has %zu floats, expected %zu", n_floats, want);
  PBG_CUDA(c, cudaSetDevice(c->dims.device));
  c->d_loaded = false;
  const float* w1 = p;            const float* b1 = w1 + H * K0;
  const float* w2 = b1 + H;       const float* b2 = w2 + H2 * H;
  const float* w3 = b2 + H2;      const float* b3 = w3 + H2;
  PBG_TRY(upload_linear(c, c->d[0], (int)H, (int)K0, c->kd0p, w1, b1));
  PBG_TRY(upload_linear(c, c->d[1], (int)H2, (int)H, c->hdp, w2, b2));
  cudaFree(c->d_w3); cudaFree(c->d_w3_pad); c->d_w3 = c->d_w3_pad = nullptr;
  const int np = c->d[1].np;  // the row-dot walks the padded width of layer 2
  PBG_CUDA(c, cudaMalloc(&c->d_w3, sizeof(float) * H2));
  PBG_CUDA(c, cudaMalloc(&c->d_w3_pad, sizeof(float) * np));
  PBG_CUDA(c, cudaMemcpyAsync(c->d_w3, w3, sizeof(float) * H2, cudaMemcpyHostToDevice, c->own_stream));
  { LaunchScope ls(c, PBG_K_OTHER, c->own_stream);
    pad_f32_kernel<<<8, 256, 0, c->own_stream>>>(c->d_w3, c->d_w3_pad, (int)H2, np); }
  PBG_CUDA(c, cudaGetLastError());
  PBG_CUDA(c, cudaStreamSynchronize(c->own_stream));
  c->d_b3 = *b3;
  c->d_loaded = true;
  return PBG_OK;
}

int pbg_generator_forward(pbg_ctx* c, const float* h, const float* r, const float* z, void* out, int64_t B,
                          int precision, int out_dtype, void* stream) {
  if (!c) return PBG_ERR_INVALID;
  if (B > 0 && (!h || !r || !out)) return fail(c, PBG_ERR_INVALID, "null tensor");
  Pass a; a.h = h; a.r = r; a.z = z; a.gen_out = out; a.out_dtype = out_dtype; a.run_g = true;
  a.B = B; a.prec = precision; a.stream = (cudaStream_t)stream;
  return run_pass(c, a);
}

int pbg_generator_forward_gather(pbg_ctx* c, const float* node_emb, int64_t N, const float* rel_emb, int64_t R,
                                 const int64_t* heads, int64_t head_stride, const int64_t* rels, int64_t rel_stride,
                                 const float* z, void* out, int64_t B, int precision, int out_dtype, void* stream) {
  if (!c) return PBG_ERR_INVALID;
  if (B > 0 && (!node_emb || !rel_emb || !heads || !rels || !out)) return fail(c, PBG_ERR_INVALID, "null tensor");
  Pass a; a.node_emb = node_emb; a.N = N; a.rel_emb = rel_emb; a.R = R;
  a.heads = (const long long*)heads; a.hs = head_stride; a.rels = (const long long*)rels; a.rs = rel_stride;
  a.z = z; a.gen_out = out; a.out_dtype = out_dtype; a.run_g = true;
  a.B = B; a.prec = precision; a.stream = (cudaStream_t)stream;
  return run_pass(c, a);
}

int pbg_discriminator_forward(pbg_ctx* c, const float* h, const float* r, const float* t, float* logits, float* probs,
                              int64_t B, int precision, void* stream) {
  if (!c) return PBG_ERR_INVALID;
  if (B > 0 && (!h || !r || !t || !logits)) return fail(c, PBG_ERR_INVALID, "null tensor");
  Pass a; a.h = h; a.r = r; a.t = t; a.logits = logits; a.probs = probs; a.run_d = true;
  a.B = B; a.prec = precision; a.stream = (cudaStream_t)stream;
  return run_pass(c, a);
}

int pbg_discriminator_score_triplets(pbg_ctx* c, const float* node_emb, int64_t N, const float* rel_emb, int64_t R,
                                     const int64_t* triplets, float* logits, float* probs, int64_t B, int precision,
                                     void* stream) {
  return pbg_score_triplets(c, node_emb, N, rel_emb, R, triplets, nullptr, nullptr, PBG_DT_F32, nullptr, logits, probs,
                            B, precision, stream);
}

int pbg_score_triplets(pbg_ctx* c, const float* node_emb, int64_t N, const float* rel_emb, int64_t R,
                       const int64_t* triplets, const float* z, void* gen_out, int out_dtype, float* gen_scores,
                       float* logits, float* probs, int64_t B, int precision, void* stream) {
  if (!c) return PBG_ERR_INVALID;
  if (B > 0 && (!node_emb || !rel_emb || !triplets)) return fail(c, PBG_ERR_INVALID, "null tensor");
  Pass a; a.node_emb = node_emb; a.N = N; a.rel_emb = rel_emb; a.R = R;
  const long long* t = (const long long*)triplets;
  a.heads = t; a.rels = t + 1; a.tails = t + 2; a.hs = a.rs = a.ts = 3;
  a.z = z; a.gen_out = gen_out; a.out_dtype = out_dtype; a.gen_scores = gen_scores;
  a.logits = logits; a.probs = probs;
  a.run_g = (gen_out != nullptr || gen_scores != nullptr); a.run_d = (logits != nullptr);
  a.B = B; a.prec = precision; a.stream = (cudaStream_t)stream;
  return run_pass(c, a);
}

int pbg_reserve(pbg_ctx* c, int64_t rows, int precision, int stage_slots) {
  if (!c) return PBG_ERR_INVALID;
  if (rows <= 0) return fail(c, PBG_ERR_INVALID, "reserve: rows must be positive");
  if (precision != PBG_PREC_F32 && precision != PBG_PREC_BF16) return fail(c, PBG_ERR_INVALID, "unknown precision %d", precision);
  if (stage_slots < 0 || stage_slots > 2) return fail(c, PBG_ERR_INVALID, "reserve: stage_slots must be 0, 1 or 2");
  PBG_CUDA(c, cudaSetDevice(c->dims.device));
  const long long chunk = std::min<long long>(rows, kMaxChunk);
  PBG_TRY(ensure_ws(c, precision, chunk, nullptr));
  PBG_TRY(ensure_latents(c, chunk, nullptr));
  for (int i = 0; i < stage_slots; ++i) PBG_TRY(ensure_stage(c, c->stage[i], chunk, nullptr));
  return PBG_OK;
}

int pbg_draw_latents(pbg_ctx* c, uint64_t seed, uint64_t offset, int64_t total_rows, int64_t row_begin, int64_t rows,
                     float* z_out, uint64_t* offset_after, void* stream) {
  if (!c) return PBG_ERR_INVALID;
  PBG_TRY(check_draw_size(c, total_rows));
  if (row_begin < 0 || rows < 0 || row_begin + rows > total_rows)
    return fail(c, PBG_ERR_INVALID, "latent draw: rows [%lld, %lld) outside the %lld of the draw", (long long)row_begin,
                (long long)(row_begin + rows), (long long)total_rows);
  if (rows > 0 && !z_out) return fail(c, PBG_ERR_INVALID, "null tensor");
  if (offset % 4) return fail(c, PBG_ERR_INVALID, "latent draw: the Philox offset must be a multiple of 4, as torch's");
  PBG_CUDA(c, cudaSetDevice(c->dims.device));
  PBG_TRY(launch_draw(c, seed, offset, nullptr, false, total_rows, row_begin, rows, z_out, (cudaStream_t)stream));
  if (offset_after)
    *offset_after = offset + latent_geometry(total_rows * c->dims.noise_dim, c->num_sms, c->max_threads_sm).inc;
  return PBG_OK;
}

int pbg_set_latent_stream(pbg_ctx* c, int enable, uint64_t seed, uint64_t offset) {
  if (!c) return PBG_ERR_INVALID;
  if (offset % 4) return fail(c, PBG_ERR_INVALID, "latent stream: the Philox offset must be a multiple of 4, as torch's");
  PBG_CUDA(c, cudaSetDevice(c->dims.device));
  PBG_CUDA(c, cudaDeviceSynchronize());   // no draw of the ctx may still be reading or advancing the offset
  const LatentStream st{offset, 0u};
  PBG_CUDA(c, cudaMemcpy(c->lat_st, &st, sizeof st, cudaMemcpyHostToDevice));
  c->lat_on = enable != 0;
  c->lat_seed = seed;
  return PBG_OK;
}

int pbg_get_latent_stream(pbg_ctx* c, uint64_t* seed, uint64_t* offset, void* stream) {
  if (!c || !seed || !offset) return PBG_ERR_INVALID;
  PBG_CUDA(c, cudaSetDevice(c->dims.device));
  LatentStream st{};
  PBG_CUDA(c, cudaMemcpyAsync(&st, c->lat_st, sizeof st, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  PBG_CUDA(c, cudaStreamSynchronize((cudaStream_t)stream));
  *seed = c->lat_seed;
  *offset = st.offset;
  return PBG_OK;
}

namespace {
// The gather of a [B, 3] triplet request into staging slot `st`: the generator's first-layer rows (when `gen`) and the
// discriminator's (when `disc`).
GatherParams slot_gather(const pbg_ctx* c, const StageSlot& st, const float* node_emb, long long N, const float* rel_emb,
                         long long R, const long long* t, const float* z, long long B, bool gen, bool disc) {
  GatherParams gp{};
  gp.node_emb = node_emb; gp.rel_emb = rel_emb; gp.N = N; gp.R = R; gp.E = c->dims.embed_dim; gp.Z = c->dims.noise_dim;
  gp.heads = t; gp.rels = t + 1; gp.tails = t + 2; gp.head_stride = gp.rel_stride = gp.tail_stride = 3;
  gp.z = z;
  gp.xg = gen ? st.xg0 : nullptr; gp.ldg = c->kg0p;
  gp.xd = disc ? st.xd0 : nullptr; gp.ldd = c->kd0p;
  gp.B = B; gp.err_flag = c->err_flag;
  return gp;
}

// The pass over staged slot `slot` that produces the requested results; the slot must hold the operands they need.
int staged_pass(pbg_ctx* c, int slot, void* gen_out, int out_dtype, float* gen_scores, float* logits, float* probs,
                void* stream, Pass& a) {
  if (slot < 0 || slot > 1) return fail(c, PBG_ERR_INVALID, "score_staged: slot must be 0 or 1");
  const StageSlot& st = c->stage[slot];
  if (st.B <= 0) return fail(c, PBG_ERR_INVALID, "score_staged: nothing staged in slot %d", slot);
  a.gen_out = gen_out; a.out_dtype = out_dtype; a.gen_scores = gen_scores; a.logits = logits; a.probs = probs;
  a.run_g = (gen_out != nullptr || gen_scores != nullptr); a.run_d = (logits != nullptr);
  if (a.run_g && !st.has_g) return fail(c, PBG_ERR_INVALID, "score_staged: slot %d holds no generator operands", slot);
  if (a.run_d && !st.has_d) return fail(c, PBG_ERR_INVALID, "score_staged: slot %d holds no discriminator operands", slot);
  a.B = st.B; a.prec = PBG_PREC_BF16; a.stream = (cudaStream_t)stream;
  return PBG_OK;
}
}  // namespace

int pbg_stage_triplets(pbg_ctx* c, int slot, const float* node_emb, int64_t N, const float* rel_emb, int64_t R,
                       const int64_t* triplets, const float* z, int64_t B, int want_gen, int want_disc, void* stream) {
  if (!c) return PBG_ERR_INVALID;
  if (slot < 0 || slot > 1) return fail(c, PBG_ERR_INVALID, "stage: slot must be 0 or 1");
  if (B <= 0 || B > kMaxChunk) return fail(c, PBG_ERR_INVALID, "stage: B must be in [1, %lld]", kMaxChunk);
  if (!node_emb || !rel_emb || !triplets) return fail(c, PBG_ERR_INVALID, "null tensor");
  if (!want_gen && !want_disc) return fail(c, PBG_ERR_INVALID, "stage: nothing to stage");
  if (want_gen && !c->g_loaded) return fail(c, PBG_ERR_NOT_LOADED, "generator weights not loaded");
  if (want_disc && !c->d_loaded) return fail(c, PBG_ERR_NOT_LOADED, "discriminator weights not loaded");
  if (want_gen && !z && !c->lat_on) return fail(c, PBG_ERR_INVALID, "generator needs latents z");
  PBG_CUDA(c, cudaSetDevice(c->dims.device));
  cudaStream_t s = (cudaStream_t)stream;
  StageSlot& st = c->stage[slot];
  PBG_TRY(ensure_stage(c, st, B, s));
  if (want_gen && !z) {   // the request's latents from the ctx's stream, in staging order
    PBG_TRY(draw_stream(c, B, st.z, s));
    z = st.z;
  }
  const long long* t = (const long long*)triplets;
  StageParams sp{};
  sp.g = slot_gather(c, st, node_emb, N, rel_emb, R, t, z, B, want_gen != 0, want_disc != 0);
  sp.xt = want_gen ? st.xt : nullptr;
  const int blocks = (int)std::min<long long>((B + 3) / 4, (long long)c->num_sms * 16);
  { LaunchScope ls(c, PBG_K_GATHER, s);
    stage_rows_kernel<<<blocks, 128, 0, s>>>(sp); }
  PBG_CUDA(c, cudaGetLastError());
  st.B = B; st.has_g = want_gen != 0; st.has_d = want_disc != 0; st.has_xt = want_gen != 0;
  st.node_emb = node_emb; st.N = N; st.tails = t + 2;
  return PBG_OK;
}

int pbg_score_staged(pbg_ctx* c, int slot, void* gen_out, int out_dtype, float* gen_scores, float* logits, float* probs,
                     void* stream) {
  if (!c) return PBG_ERR_INVALID;
  Pass a;
  PBG_TRY(staged_pass(c, slot, gen_out, out_dtype, gen_scores, logits, probs, stream, a));
  if (!a.run_g && !a.run_d) return PBG_OK;
  PBG_CUDA(c, cudaSetDevice(c->dims.device));
  PBG_TRY(ensure_ws(c, PBG_PREC_BF16, a.B, a.stream));
  GatherParams gp{};
  return launch_pass2(c, c->ws_bf16, a, gp, 0, a.B, gen_out, gen_scores, true, &c->stage[slot]);
}

int pbg_score_staged_stage_next(pbg_ctx* c, int slot, void* gen_out, int out_dtype, float* gen_scores, float* logits, float* probs,
                                const float* node_emb, int64_t N, const float* rel_emb, int64_t R, const int64_t* next_triplets,
                                const float* next_z, int64_t next_B, void* stream) {
  if (!c) return PBG_ERR_INVALID;
  Pass a;
  PBG_TRY(staged_pass(c, slot, gen_out, out_dtype, gen_scores, logits, probs, stream, a));
  StageSlot& st = c->stage[slot];
  StageSlot& nx = c->stage[1 - slot];
  if (next_B <= 0 || next_B > kMaxChunk) return fail(c, PBG_ERR_INVALID, "stage next: B must be in [1, %lld]", kMaxChunk);
  if (!node_emb || !rel_emb || !next_triplets) return fail(c, PBG_ERR_INVALID, "null tensor");
  if (!a.run_g && !a.run_d) return fail(c, PBG_ERR_INVALID, "score_staged_stage_next: no result requested");
  if (a.run_g && !next_z && !c->lat_on) return fail(c, PBG_ERR_INVALID, "generator needs latents z");
  PBG_CUDA(c, cudaSetDevice(c->dims.device));
  PBG_TRY(ensure_ws(c, PBG_PREC_BF16, a.B, a.stream));
  PBG_TRY(ensure_stage(c, nx, next_B, a.stream));
  if (a.run_g && !next_z) {   // drawn now, ahead of the pass that gathers it: stream order is staging order
    PBG_TRY(draw_stream(c, next_B, nx.z, a.stream));
    next_z = nx.z;
  }
  // the next request gets the operands this pass produces results for (same models in flight)
  const long long* t = reinterpret_cast<const long long*>(next_triplets);
  const GatherParams gp = slot_gather(c, nx, node_emb, N, rel_emb, R, t, next_z, next_B, a.run_g, a.run_d);
  PBG_TRY(launch_pass2(c, c->ws_bf16, a, gp, 0, a.B, gen_out, gen_scores, true, &st, true));
  st.B = -1;   // consumed (with the workspace discard on its rows are dropped from L2 as the first layers finish with them)
  nx.B = next_B; nx.has_g = a.run_g; nx.has_d = a.run_d; nx.has_xt = false;
  nx.node_emb = node_emb; nx.N = N; nx.tails = t + 2;
  return PBG_OK;
}

int pbg_linear_bf16(pbg_ctx* c, int model, int layer, const void* a, void* out, int64_t M, void* stream) {
  if (!c || !a || !out || M <= 0) return c ? fail(c, PBG_ERR_INVALID, "bad argument") : PBG_ERR_INVALID;
  if (model == 0 && !c->g_loaded) return fail(c, PBG_ERR_NOT_LOADED, "generator weights not loaded");
  if (model == 1 && !c->d_loaded) return fail(c, PBG_ERR_NOT_LOADED, "discriminator weights not loaded");
  if (model < 0 || model > 1 || layer < 0 || layer > (model == 0 ? 2 : 1)) return fail(c, PBG_ERR_INVALID, "no such layer");
  if (M > kMaxChunk) return fail(c, PBG_ERR_INVALID, "linear_bf16: at most %lld rows", kMaxChunk);
  PBG_CUDA(c, cudaSetDevice(c->dims.device));
  cudaStream_t s = (cudaStream_t)stream;
  PBG_TRY(ensure_ws(c, PBG_PREC_BF16, M, s));
  Workspace& w = c->ws_bf16;
  // ONE layer of the product kernel: the pass kernel with a single item kind, its A operand the caller's matrix and no
  // dependency to wait for; the layer's own epilogue (LeakyReLU store / row dot + sigmoid / tanh) writes `out`.
  static const int kind_of[2][3] = {{IT_G_L0, IT_G_L1, IT_G_L2}, {IT_D_L0, IT_D_L1, -1}};
  const int k = kind_of[model][layer];
  const Linear& l = model == 0 ? c->g[layer] : c->d[layer];
  const bool store = kEpiOf[k] == PEPI_STORE;
  CUtensorMap amap, omap;
  PBG_TRY(make_tmap(c, &amap, a, M, l.kp, kBlockM));
  if (store) PBG_TRY(make_tmap(c, &omap, out, M, l.np, 32));
  Pass2Params p;
  memset(&p, 0, sizeof p);
  set_layer(p, k, l, amap, store ? &omap : nullptr, store ? static_cast<__nv_bfloat16*>(out) : nullptr, l.np);
  const int nrb = static_cast<int>((M + kP2Rows - 1) / kP2Rows);
  p.seg[0] = P2Segment{k, p.layer[k].n_tiles, 0, 0, k, 0};
  p.n_seg = 1; p.n_total = nrb * p.layer[k].n_tiles;
  p.no_deps = 1; p.gather_external = 1; p.phase0_groups = 0;
  p.poll_ns = 40; p.gather_defer = 1;
  p.nrb = nrb; p.rb_cap = w.mb_cap; p.M = static_cast<int>(M); p.slope = c->dims.leaky_slope;
  p.sched = w.sched; p.ready = w.ready; p.fin = w.fin;
  p.part_g = w.part_g; p.part_d = w.part_d;
  if (k == IT_G_L2) {
    p.gen_out = out; p.out_f32 = 1; p.n_valid = c->dims.embed_dim; p.ld_gen = c->dims.embed_dim;
    p.slots_g = (c->dims.embed_dim + 63) / 64;
  }
  if (k == IT_D_L1) {
    if (l.np / 64 > kPartSlotsD) return fail(c, PBG_ERR_UNSUPPORTED, "d_hidden too wide for the partial buffer");
    p.w3 = c->d_w3_pad; p.b3 = c->d_b3; p.logits = static_cast<float*>(out); p.slots_d = l.np / 64;
  }
  p.w3_off = -1;   // biases / final dot weights through the global path (BIASS = false instantiation)
  const int grid = pass_grid(c) & ~1;
  cudaError_t le;
  { LaunchScope ls(c, model == 0 ? PBG_K_G_L0 + layer : PBG_K_D_L0 + layer, s);
    le = launch_pdl(false, kPass2[0], grid, kP2Threads, P2Smem::kTotal, s, p); }
  if (le == cudaSuccess) le = cudaGetLastError();
  if (le != cudaSuccess) return fail(c, PBG_ERR_CUDA, "single-layer pass launch failed: %s", cudaGetErrorString(le));
  return PBG_OK;
}

int pbg_profile_enable(pbg_ctx* c, int enable) {
  if (!c) return PBG_ERR_INVALID;
  c->profiling = enable != 0;
  return PBG_OK;
}

int pbg_profile_read(pbg_ctx* c, double* ms, int64_t* count) {
  if (!c || !ms || !count) return PBG_ERR_INVALID;
  PBG_CUDA(c, cudaSetDevice(c->dims.device));
  PBG_CUDA(c, cudaDeviceSynchronize());
  for (auto& r : c->prof) {
    float t = 0.f;
    if (cudaEventElapsedTime(&t, r.a, r.b) == cudaSuccess && r.kind >= 0 && r.kind < PBG_NUM_KERNEL_KINDS) {
      ms[r.kind] += t; count[r.kind] += 1;
    }
    cudaEventDestroy(r.a); cudaEventDestroy(r.b);
  }
  c->prof.clear();
  return PBG_OK;
}

int pbg_debug_trace(pbg_ctx* c, int enable, int64_t* host_out, int64_t n_slots) {
  if (!c) return PBG_ERR_INVALID;
  PBG_CUDA(c, cudaSetDevice(c->dims.device));
  PBG_CUDA(c, cudaDeviceSynchronize());
  const size_t n = static_cast<size_t>(c->num_sms) * kTraceSlots;
  if (host_out && c->trace) {
    std::vector<long long> tmp(n);
    PBG_CUDA(c, cudaMemcpy(tmp.data(), c->trace, n * sizeof(long long), cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < n && i < static_cast<size_t>(n_slots); ++i) host_out[i] = tmp[i];
  }
  if (enable && !c->trace) {
    PBG_CUDA(c, cudaMalloc(&c->trace, n * sizeof(long long)));
  } else if (!enable && c->trace) {
    cudaFree(c->trace); c->trace = nullptr;
  }
  if (c->trace) PBG_CUDA(c, cudaMemset(c->trace, 0, n * sizeof(long long)));
  return PBG_OK;
}

int pbg_check_indices(pbg_ctx* c, void* stream) {
  if (!c) return PBG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PBG_CUDA(c, cudaSetDevice(c->dims.device));
  PBG_CUDA(c, cudaMemcpyAsync(c->err_flag_host, c->err_flag, sizeof(int), cudaMemcpyDeviceToHost, s));
  if (c->host_block) {
    // PBG_HOST_SYNC=block: the calling thread sleeps until the stream has drained instead of spinning on it -- for hosts
    // with fewer cores than synchronous callers (8 ranks x 6 threads on 32 cores); costs a wake-up latency per call
    if (!c->host_evt) PBG_CUDA(c, cudaEventCreateWithFlags(&c->host_evt, cudaEventBlockingSync | cudaEventDisableTiming));
    PBG_CUDA(c, cudaEventRecord(c->host_evt, s));
    PBG_CUDA(c, cudaEventSynchronize(c->host_evt));
  } else {
    PBG_CUDA(c, cudaStreamSynchronize(s));
  }
  if (*c->err_flag_host != 0) {
    PBG_CUDA(c, cudaMemsetAsync(c->err_flag, 0, sizeof(int), s));
    PBG_CUDA(c, cudaStreamSynchronize(s));
    return fail(c, PBG_ERR_INDEX, "index out of range in embedding gather");
  }
  return PBG_OK;
}

namespace {
// Shared body of the *_host entry points.  packed: the caller's buffers are TWO blocks -- in_block = [triplets int64
// B x 3 | z fp32 B x Z], out_block = [gen_scores | logits | probs] fp32 B each -- and travel in one copy per direction.
int score_host(pbg_ctx* c, const float* node_emb, int64_t N, const float* rel_emb, int64_t R, const int64_t* triplets_host,
               const float* z_host, float* gen_out_host, float* gen_scores_host, float* logits_host, float* probs_host,
               int64_t B, int precision, bool packed) {
  if (!c) return PBG_ERR_INVALID;
  if (B < 0) return fail(c, PBG_ERR_INVALID, "negative batch");
  if (B == 0) return PBG_OK;
  if (!triplets_host) return fail(c, PBG_ERR_INVALID, "null triplets");
  const bool run_g = gen_out_host || gen_scores_host;
  if (run_g && !z_host && !c->lat_on) return fail(c, PBG_ERR_INVALID, "generator needs latents z");
  PBG_CUDA(c, cudaSetDevice(c->dims.device));
  const int E = c->dims.embed_dim, Z = c->dims.noise_dim;
  cudaStream_t s = c->own_stream;
  if (c->host_cap < B) {
    PBG_TRY(begin_growth(c, s, "the host staging block"));
    c->host_cap = 0;
    const size_t per_row = sizeof(long long) * 3 + sizeof(float) * (Z + 3 + E);
    PBG_TRY(realloc_dev(c, c->st_block, per_row * B + 64));   // + alignment padding in front of z and gen_out
    c->host_cap = B;
  }
  // one device block, laid out for THIS call's B: [triplets | z | scores | logits | probs | gen_out]; z and gen_out rows
  // are read / written with 16-byte vectors, so their offsets are rounded up
  auto up16 = [](size_t v) { return (v + 15) & ~static_cast<size_t>(15); };
  char* b0 = c->st_block;
  size_t off = 0;
  long long* trip = reinterpret_cast<long long*>(b0 + off);  off = up16(off + sizeof(long long) * 3 * B);
  float* z = reinterpret_cast<float*>(b0 + off);             off += sizeof(float) * Z * B;
  float* scores = reinterpret_cast<float*>(b0 + off);        off += sizeof(float) * B;
  float* logits = reinterpret_cast<float*>(b0 + off);        off += sizeof(float) * B;
  float* probs = reinterpret_cast<float*>(b0 + off);         off = up16(off + sizeof(float) * B);
  float* gen = reinterpret_cast<float*>(b0 + off);
  // every DMA operation costs a few microseconds of set-up beside its bytes (six of them were a third of a 4096-triplet
  // call): the packed form moves [triplets | z] and [scores | logits | probs] in one copy each
  const bool one_h2d = packed && z_host && reinterpret_cast<char*>(z) == reinterpret_cast<char*>(trip) + sizeof(long long) * 3 * B;
  if (one_h2d) {
    PBG_CUDA(c, cudaMemcpyAsync(trip, triplets_host, sizeof(long long) * 3 * B + sizeof(float) * Z * B, cudaMemcpyHostToDevice, s));
  } else {
    PBG_CUDA(c, cudaMemcpyAsync(trip, triplets_host, sizeof(long long) * 3 * B, cudaMemcpyHostToDevice, s));
    if (run_g && z_host) PBG_CUDA(c, cudaMemcpyAsync(z, z_host, sizeof(float) * Z * B, cudaMemcpyHostToDevice, s));
  }
  PBG_TRY(pbg_score_triplets(c, node_emb, N, rel_emb, R, (const int64_t*)trip, run_g && z_host ? z : nullptr,
                             gen_out_host ? gen : nullptr, PBG_DT_F32, gen_scores_host ? scores : nullptr,
                             logits_host ? logits : nullptr, probs_host ? probs : nullptr, B, precision, s));
  if (packed) {
    PBG_CUDA(c, cudaMemcpyAsync(gen_scores_host, scores, sizeof(float) * 3 * B, cudaMemcpyDeviceToHost, s));
  } else {
    if (gen_scores_host) PBG_CUDA(c, cudaMemcpyAsync(gen_scores_host, scores, sizeof(float) * B, cudaMemcpyDeviceToHost, s));
    if (logits_host) PBG_CUDA(c, cudaMemcpyAsync(logits_host, logits, sizeof(float) * B, cudaMemcpyDeviceToHost, s));
    if (probs_host) PBG_CUDA(c, cudaMemcpyAsync(probs_host, probs, sizeof(float) * B, cudaMemcpyDeviceToHost, s));
  }
  if (gen_out_host) PBG_CUDA(c, cudaMemcpyAsync(gen_out_host, gen, sizeof(float) * E * B, cudaMemcpyDeviceToHost, s));
  return pbg_check_indices(c, s);  // one sync: results + the out-of-range flag
}
}  // namespace

int pbg_score_triplets_host(pbg_ctx* c, const float* node_emb, int64_t N, const float* rel_emb, int64_t R,
                            const int64_t* triplets_host, const float* z_host, float* gen_out_host,
                            float* gen_scores_host, float* logits_host, float* probs_host, int64_t B, int precision) {
  return score_host(c, node_emb, N, rel_emb, R, triplets_host, z_host, gen_out_host, gen_scores_host, logits_host, probs_host, B,
                    precision, false);
}

int pbg_score_triplets_host_packed(pbg_ctx* c, const float* node_emb, int64_t N, const float* rel_emb, int64_t R,
                                   const void* in_block_host, float* out_block_host, int64_t B, int precision) {
  if (!c) return PBG_ERR_INVALID;
  if (B > 0 && (!in_block_host || !out_block_host)) return fail(c, PBG_ERR_INVALID, "null block");
  const int64_t* trip = static_cast<const int64_t*>(in_block_host);
  const float* z = reinterpret_cast<const float*>(static_cast<const char*>(in_block_host) + sizeof(long long) * 3 * B);
  return score_host(c, node_emb, N, rel_emb, R, trip, z, nullptr, out_block_host, out_block_host + B, out_block_host + 2 * B, B,
                    precision, true);
}

int pbg_score_triplets_host_ids(pbg_ctx* c, const float* node_emb, int64_t N, const float* rel_emb, int64_t R,
                                const int64_t* triplets_host, float* out_block_host, int64_t B, int precision) {
  if (!c) return PBG_ERR_INVALID;
  if (!c->lat_on) return fail(c, PBG_ERR_INVALID, "score_triplets_host_ids draws the latents: enable the latent stream first");
  if (B > 0 && (!triplets_host || !out_block_host)) return fail(c, PBG_ERR_INVALID, "null block");
  return score_host(c, node_emb, N, rel_emb, R, triplets_host, nullptr, nullptr, out_block_host, out_block_host + B,
                    out_block_host + 2 * B, B, precision, true);
}

}  // extern "C"
