/* pbg.h -- C ABI of libpbg_b200.so: the B200 (sm_100a) replacement for the one hot path of
 * Drjay806/PRO-B-GAN: the generator forward pass and the discriminator scoring pass that
 * pro_b_gan_infer.py drives.  Citations are file:line into the reference.
 *
 * Conventions
 *   - every function returns a pbg_status (0 = OK); no C++ exception crosses the ABI;
 *     pbg_last_error() gives the message for the last non-zero status.
 *   - all tensor pointers are DEVICE pointers on the ctx's device unless the name ends in
 *     _host; buffers are caller-owned, row-major and contiguous; fp32 unless stated.
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).  Device-pointer
 *     entry points are stream-ordered and never synchronise; *_host entry points are
 *     synchronous (H2D copy, kernels, D2H copy, one stream sync).
 *   - a ctx is bound to one device and is not thread-safe (the reference is single
 *     threaded and synchronous, pro_b_gan_infer.py:133-165).
 *   - there is no CPU fallback: on a machine without an sm_100 device pbg_create fails.
 */
#ifndef PBG_H_
#define PBG_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PBG_ABI_VERSION 1

typedef struct pbg_ctx pbg_ctx;

typedef enum pbg_status {
  PBG_OK = 0,
  PBG_ERR_INVALID = 1,     /* bad argument / shape                                        */
  PBG_ERR_CUDA = 2,        /* a CUDA runtime or driver call failed                        */
  PBG_ERR_NOT_LOADED = 3,  /* forward called before the matching pbg_load_*               */
  PBG_ERR_INDEX = 4,       /* an entity / relation id was out of range (-> IndexError)    */
  PBG_ERR_UNSUPPORTED = 5, /* no sm_100 device, or dims the kernels cannot tile           */
  PBG_ERR_NOMEM = 6
} pbg_status;

/* arithmetic mode of the Linear layers */
typedef enum pbg_precision {
  PBG_PREC_F32 = 0,  /* SIMT FFMA, fp32 end to end: the parity mode (max-abs 1e-4)        */
  PBG_PREC_BF16 = 1  /* tcgen05 kind::f16 (bf16 x bf16 -> fp32 in TMEM): the fast mode    */
} pbg_precision;

/* element type of the generator output buffer */
typedef enum pbg_dtype { PBG_DT_F32 = 0, PBG_DT_BF16 = 1 } pbg_dtype;

/* Model dimensions.  embed_dim / noise_dim / d_hidden are the checkpoint's args
 * (pro_b_gan_infer.py:77-80); g_hidden is the generator's internal hidden width (the
 * reference passes no hidden_dim to Generator, :93; the oracle default is 1024). */
typedef struct pbg_dims {
  int32_t embed_dim;  /* E */
  int32_t noise_dim;  /* Z */
  int32_t g_hidden;   /* generator: (2E+Z) -> g_hidden -> g_hidden -> E                   */
  int32_t d_hidden;   /* discriminator: 3E -> d_hidden -> d_hidden/2 -> 1                 */
  int32_t device;     /* CUDA device ordinal                                              */
  float leaky_slope;  /* LeakyReLU negative slope (0.2)                                   */
} pbg_dims;

int pbg_abi_version(void);

/* Replaces `Generator(E, Z).to(device)` / `Discriminator(E, H).to(device)`
 * (pro_b_gan_infer.py:93-94): allocates the device-side state for one model pair.
 * Accepts embed_dim, noise_dim and g_hidden that are multiples of 8, d_hidden a multiple of 16 and
 * leaky_slope in [0, 1]; anything else is PBG_ERR_UNSUPPORTED.  bf16 mode has two further limits,
 * checked at launch (PBG_ERR_UNSUPPORTED, the ctx stays usable): a pass that runs the generator needs
 * embed_dim <= 512, and a pass that runs the discriminator needs d_hidden <= 8192 (d_hidden / 2
 * rounded up to 128 is at most 4096).  fp32 mode has neither limit. */
int pbg_create(pbg_ctx** out, const pbg_dims* dims);
void pbg_destroy(pbg_ctx* ctx);

/* Message for the last failing call on ctx (ctx == NULL: last failing pbg_create). */
const char* pbg_last_error(const pbg_ctx* ctx);

/* Replaces `generator.load_state_dict(...)` + `.eval()` (pro_b_gan_infer.py:97, :106).
 * `packed_host` is a HOST buffer of fp32 with eval-mode BatchNorm already folded into the
 * preceding Linear by the host (legal because of :106 / torch.no_grad :133):
 *   W1[g_hidden, 2E+Z] b1[g_hidden] W2[g_hidden, g_hidden] b2[g_hidden] W3[E, g_hidden] b3[E]
 * (each W row-major [out, in], PyTorch's nn.Linear layout).  n_floats must match exactly. */
int pbg_load_generator(pbg_ctx* ctx, const float* packed_host, size_t n_floats);

/* Replaces `discriminator.load_state_dict(...)` + `.eval()` (pro_b_gan_infer.py:98, :107):
 *   W1[H, 3E] b1[H] W2[H/2, H] b2[H/2] w3[H/2] b3[1] */
int pbg_load_discriminator(pbg_ctx* ctx, const float* packed_host, size_t n_floats);

/* Replaces `self.generator(h_emb, r_emb)` (pro_b_gan_infer.py:143, :201).
 * h, r: [B,E] fp32; z: [B,Z] fp32 latents (the reference's forward takes no noise argument;
 * the host module draws z from its seeded CPU generator and passes it here; NULL draws from the ctx's latent
 * stream, see pbg_set_latent_stream).
 * out: [B,E] of `out_dtype`.  tanh output. */
int pbg_generator_forward(pbg_ctx* ctx, const float* h, const float* r, const float* z, void* out,
                          int64_t B, int precision, int out_dtype, void* stream);

/* Replaces gather + forward: `h_emb = node_emb[heads]; r_emb = rel_emb(relations);
 * generator(h_emb, r_emb)` (pro_b_gan_infer.py:139-143 and :186-187, :201).
 * node_emb [N,E], rel_emb [R,E]; heads / rels are int64 with element strides (the
 * reference's `triplet_tensor[:, i]` columns are stride-3 views, :183). */
int pbg_generator_forward_gather(pbg_ctx* ctx, const float* node_emb, int64_t N, const float* rel_emb,
                                 int64_t R, const int64_t* heads, int64_t head_stride,
                                 const int64_t* rels, int64_t rel_stride, const float* z, void* out,
                                 int64_t B, int precision, int out_dtype, void* stream);

/* Replaces `self.discriminator(h_emb, r_emb, t_emb)` (pro_b_gan_infer.py:301) and the
 * sigmoid that follows it (:302).  logits [B] fp32; probs [B] fp32 or NULL. */
int pbg_discriminator_forward(pbg_ctx* ctx, const float* h, const float* r, const float* t,
                              float* logits, float* probs, int64_t B, int precision, void* stream);

/* Replaces `discriminator.score_triplets(node_emb, rel_emb, triplet_tensor)`
 * (pro_b_gan_infer.py:207): triplets [B,3] int64 contiguous (head, relation, tail). */
int pbg_discriminator_score_triplets(pbg_ctx* ctx, const float* node_emb, int64_t N,
                                     const float* rel_emb, int64_t R, const int64_t* triplets,
                                     float* logits, float* probs, int64_t B, int precision,
                                     void* stream);

/* The canonical generator+discriminator pass of `ProtBGANInference.score_triplets`
 * (pro_b_gan_infer.py:186-188, :201-202, :207) in one call sharing one gather:
 *   gen_out    [B,E] predicted tail embeddings (G.forward, :201), or NULL
 *   gen_scores [B]   cosine_similarity(pred, node_emb[tail], dim=1) (:202), or NULL
 *                    (both NULL: the generator is skipped)
 *   logits / probs [B] discriminator logit and sigmoid(logit) (:207); NULL logits skips D.
 * Needs the matching models loaded in this ctx. */
int pbg_score_triplets(pbg_ctx* ctx, const float* node_emb, int64_t N, const float* rel_emb, int64_t R,
                       const int64_t* triplets, const float* z, void* gen_out, int out_dtype,
                       float* gen_scores, float* logits, float* probs, int64_t B, int precision,
                       void* stream);

/* Same pass with HOST index / latent / result buffers: the end-to-end form the reference's
 * list API implies (H2D at :182, D2H at :203, :208-209).  node_emb / rel_emb stay device
 * pointers (they are model state moved once at load, :83, :102).  Synchronous.  Returns
 * PBG_ERR_INDEX if any id is out of range (results are then undefined).  Pinned (page-locked) host memory keeps
 * the copies asynchronous. */
int pbg_score_triplets_host(pbg_ctx* ctx, const float* node_emb, int64_t N, const float* rel_emb,
                            int64_t R, const int64_t* triplets_host, const float* z_host,
                            float* gen_out_host, float* gen_scores_host, float* logits_host,
                            float* probs_host, int64_t B, int precision);

/* The same call for a caller that packs a request into two host blocks (each ONE allocation):
 *   in_block_host  = [ triplets int64 B x 3 | z fp32 B x Z ]          (24 B + 4 Z B bytes)
 *   out_block_host = [ gen_scores | logits | probs ] fp32 B each      (12 B bytes)
 * Each block travels in ONE copy (a DMA operation costs microseconds of set-up beside its bytes: six of them were
 * a third of a 4096-triplet call; for an odd B the latents are not 16-byte aligned behind the triplets and the
 * inputs go in two copies).  Generator + discriminator both run.  Otherwise as pbg_score_triplets_host. */
int pbg_score_triplets_host_packed(pbg_ctx* ctx, const float* node_emb, int64_t N, const float* rel_emb,
                                   int64_t R, const void* in_block_host, float* out_block_host, int64_t B,
                                   int precision);

/* Device latents.  torch.randn((rows, Z), device='cuda', generator=g) is fully set by g's Philox (seed, offset), the
 * launch geometry of torch's normal_ and curand_normal4: element e of a draw of numel = rows * Z elements comes from
 * thread t = e % T, round r = e / 4T, component j = (e / T) % 4 with T = 256 * min(SMs * max_threads_per_SM / 256,
 * ceil(numel / 256)), and the draw advances the offset by ((numel - 1) / 4T + 1) * 4.  These calls reproduce that stream
 * bit for bit on the device (numel < 2^31; larger draws are PBG_ERR_UNSUPPORTED).  The CPU stream the host modules
 * draw from by default (mt19937) is a different stream.
 *
 * pbg_draw_latents writes rows [row_begin, row_begin + rows) of a [total_rows, Z] draw at (seed, offset) to z_out
 * [rows, Z] fp32, stream-ordered; ranges that tile [0, total_rows) concatenate to the whole draw, so a batch-sharded
 * job can draw its own shard.  *offset_after (if non-NULL) receives the offset after the whole draw.  Stateless. */
int pbg_draw_latents(pbg_ctx* ctx, uint64_t seed, uint64_t offset, int64_t total_rows, int64_t row_begin,
                     int64_t rows, float* z_out, uint64_t* offset_after, void* stream);

/* The ctx's latent stream (off by default).  While it is enabled, every entry point that runs the generator accepts
 * z == NULL (pbg_generator_forward[_gather], pbg_score_triplets, pbg_score_triplets_host with z_host == NULL,
 * pbg_stage_triplets, pbg_score_staged_stage_next with next_z == NULL) and draws the call's [B, Z] latents from
 * (seed, offset), then advances the offset as torch would: a sequence of such calls sees what the same calls given
 * z = torch.randn((B, Z), device='cuda', generator=g) see for a generator g at the same (seed, offset).
 *   - a call of B > 65536 rows (processed in chunks) draws each chunk's rows of ONE [B, Z] draw;
 *   - staged requests draw when they are staged (stream order = staging order); discriminator-only calls draw nothing;
 *   - caller-supplied latents always win and leave the stream where it was;
 *   - with the stream disabled, z == NULL is refused (PBG_ERR_INVALID) as before.
 * The offset lives in device memory and each draw kernel advances it, so a CUDA graph captured over such calls draws
 * fresh latents on every replay, as successive eager calls would; the seed is a launch argument and a graph keeps
 * the one it was captured with.  Draws from one ctx's stream must be ordered among themselves (one stream, or
 * events between an ingest and a compute stream), as the staging calls already are.  pbg_set_latent_stream
 * synchronises the device; pbg_get_latent_stream synchronises `stream` and reads the current position. */
int pbg_set_latent_stream(pbg_ctx* ctx, int enable, uint64_t seed, uint64_t offset);
int pbg_get_latent_stream(pbg_ctx* ctx, uint64_t* seed, uint64_t* offset, void* stream);

/* pbg_score_triplets_host_packed without latents on the wire: in-block = triplets int64 [B, 3] only (24 B per
 * sample), out-block = [gen_scores | logits | probs] fp32 B each (12 B per sample); the latents come from the ctx's
 * latent stream, which must be enabled (else PBG_ERR_INVALID).  Generator + discriminator both run.  Synchronous. */
int pbg_score_triplets_host_ids(pbg_ctx* ctx, const float* node_emb, int64_t N, const float* rel_emb, int64_t R,
                                const int64_t* triplets_host, float* out_block_host, int64_t B, int precision);

/* Request staging -- the ingest / compute split of the same pass for callers that keep requests in flight.
 * pbg_score_triplets does gather -> layers in one launch, so the first tiles of every pass wait for its gather.
 * A server (or bench.py) that already holds the NEXT request's ids and latents on the device can stage it while the
 * current pass runs:
 *   pbg_stage_triplets(ctx, slot, ...)  gathers + concatenates + casts the request's rows (`h = node_emb[heads]`,
 *       `rel_emb(relations)`, `node_emb[tails]`, pro_b_gan_infer.py:186-188, and the latent concat inside G) into
 *       staging slot `slot` (0 or 1) of the ctx, as a small kernel on `stream` (an ingest stream) that fits beside
 *       resident pass CTAs; want_gen / want_disc choose the operands built; B <= 65536.
 *   pbg_score_staged(ctx, slot, ...)    runs the G + D pass over the staged rows on `stream` (the compute stream);
 *       results as in pbg_score_triplets.  bf16 mode only.
 * Both are stream-ordered; the CALLER orders a slot's uses across the two streams (stage -> score -> next stage of the
 * same slot: two events, or one stream).  A ctx still runs one pass at a time.
 * pbg_reserve sizes the activation and latent workspaces (and `stage_slots` staging slots) for `rows` rows up front: buffers
 * otherwise grow lazily with a device synchronisation, which is refused (PBG_ERR_INVALID) while the stream is being
 * captured into a CUDA graph. */
int pbg_reserve(pbg_ctx* ctx, int64_t rows, int precision, int stage_slots);
int pbg_stage_triplets(pbg_ctx* ctx, int slot, const float* node_emb, int64_t N, const float* rel_emb, int64_t R,
                       const int64_t* triplets, const float* z, int64_t B, int want_gen, int want_disc, void* stream);
int pbg_score_staged(pbg_ctx* ctx, int slot, void* gen_out, int out_dtype, float* gen_scores, float* logits,
                     float* probs, void* stream);
/* pbg_score_staged for `slot` AND the staging of the next request into the other slot in ONE launch: the pass kernel's
 * epilogue warps gather the next request's rows in 4-row groups whenever they would otherwise wait for an item or an
 * accumulator, and drain what is left before they exit -- no second kernel, no second stream, nothing in the pass
 * waits for the gather.  The next request is staged with the operands of the models this call runs; its triplets (and
 * the table) must stay valid until IT has been scored (its cosine epilogue reads the tail rows through them).  A lane
 * of requests: pbg_stage_triplets(slot 0, first) once, then pbg_score_staged_stage_next(slot j & 1, ..., request j + 1)
 * per request and pbg_score_staged for the last.  The call CONSUMES the request staged in `slot` (with the workspace
 * discard on, its rows are dropped from L2 as the first layers finish with them): scoring the slot again before it
 * has been staged again is refused (PBG_ERR_INVALID); pbg_score_staged leaves a slot intact. */
int pbg_score_staged_stage_next(pbg_ctx* ctx, int slot, void* gen_out, int out_dtype, float* gen_scores, float* logits,
                                float* probs, const float* node_emb, int64_t N, const float* rel_emb, int64_t R,
                                const int64_t* next_triplets, const float* next_z, int64_t next_B, void* stream);

/* Index semantics = the reference's: head / tail ids index `node_emb` as a tensor, so -N..-1 count from the end
 * (pro_b_gan_infer.py:139, :186, :188); relation ids go through nn.Embedding, which rejects negatives (:187).
 * Out-of-range ids never fault on the device: the gather clamps them and raises a flag.
 * This synchronises `stream`, returns PBG_ERR_INDEX if the flag was raised since the last
 * check (and clears it), else PBG_OK.  The Python host turns it into IndexError, the
 * exception the reference's `node_emb[heads]` raises (pro_b_gan_infer.py:139). */
int pbg_check_indices(pbg_ctx* ctx, void* stream);

/* Diagnostics / per-layer known-answer tests: run ONE Linear layer of a loaded model on the
 * tensor cores.  model 0 = generator (layers 0..2), 1 = discriminator (layers 0..1; layer 1
 * includes the folded final H/2 -> 1 dot product).  a_bf16 is a device [M, Kp] bf16 matrix
 * (Kp = the layer's input width rounded up to 64).  out is
 *   bf16 [M, Np]  for the LeakyReLU layers (Np = output width rounded up to 128),
 *   fp32 [M, E]   for generator layer 2 (tanh),
 *   fp32 [M]      for discriminator layer 1 (logits). */
int pbg_linear_bf16(pbg_ctx* ctx, int model, int layer, const void* a_bf16, void* out, int64_t M,
                    void* stream);

/* Per-kernel device timing for bench.py's roofline: while enabled, every kernel this ctx launches is
 * bracketed by CUDA events on its launch stream.  pbg_profile_read synchronises, adds the elapsed
 * milliseconds and launch counts per kernel kind into ms[PBG_NUM_KERNEL_KINDS] /
 * count[PBG_NUM_KERNEL_KINDS], and resets the records. */
enum {
  PBG_K_GATHER = 0, /* gather + concat (+ bf16 cast)                      */
  PBG_K_G_L0 = 1,   /* generator Linear 0 (2E+Z -> H) + BN + LeakyReLU    */
  PBG_K_G_L1 = 2,   /* generator Linear 1 (H -> H) + BN + LeakyReLU       */
  PBG_K_G_L2 = 3,   /* generator Linear 2 (H -> E) + tanh (+ cosine)      */
  PBG_K_D_L0 = 4,   /* discriminator Linear 0 (3E -> H) + LeakyReLU       */
  PBG_K_D_L1 = 5,   /* discriminator Linear 1 (H -> H/2) + LeakyReLU + final dot + sigmoid */
  PBG_K_OTHER = 6,  /* fp32-mode row-dot / cosine, weight packing         */
  PBG_K_PASS = 7,   /* bf16 mode: the whole G + D pass as one persistent kernel (gather + 5 Linear layers) */
  PBG_K_TOPK = 8,   /* entity scoring + top-k: the tensor-core filter kernel                               */
  PBG_NUM_KERNEL_KINDS = 9
};
int pbg_profile_enable(pbg_ctx* ctx, int enable);
int pbg_profile_read(pbg_ctx* ctx, double* ms, int64_t* count);

/* Diagnostics: while enabled, the tensor-core kernels write clock64 slots per CTA (begin, producer / MMA /
 * epilogue wait sums, end stamps and a per-item timeline; layout in pass2_kernel.cuh) into a device buffer of
 * 256 x num_SMs slots.
 * The call synchronises the device, copies the current slots to host_out (if non-NULL, up to n_slots),
 * then enables / disables tracing and zeroes the buffer. */
int pbg_debug_trace(pbg_ctx* ctx, int enable, int64_t* host_out, int64_t n_slots);

/* Launch width of the fused pass kernel: how many CTAs (= SMs; rounded down to whole CTA pairs, at least 2) one
 * pass occupies.  0 (the default) = every SM of the device.  A 4096-triplet pass is a chain of dependent layers
 * and does not fill 148 SMs for its whole duration, so a server that has independent passes in flight gives each
 * its own ctx and stream and a width of about a third of the device: the passes then run side by side
 * (bench.py does exactly that).  One pass alone is fastest at full width. */
int pbg_set_launch_width(pbg_ctx* ctx, int n_ctas);

/* SM clock (MHz) during the last bf16-mode pass of the ctx, measured inside the kernel: CTA 0 reads clock64() and
 * %globaltimer when its roles start and when it exits.  Diagnostics for bench.py's `clocks` entry -- NVML's clock
 * reading is a sample of a much slower loop than a 50 ms timed region.  Synchronises `stream`. */
int pbg_last_pass_sm_clock(pbg_ctx* ctx, void* stream, double* mhz_out);

/* Workspace discard (default on; the environment variable PBG_DISCARD=0 turns it off for new contexts).  The layers of
 * a bf16-mode pass hand their activations to each other through L2 in workspace buffers of the ctx.  Once the
 * consuming layer has finished with a 256-row block those lines are dead but dirty, and when several contexts'
 * workspaces cycle through the L2 they are written back to HBM on eviction (32 MB per 4096-triplet pass that nothing
 * reads).  With the option on the pass kernel drops each dead block from L2 (`discard.global.L2`) instead.  Results
 * do not depend on the setting.  No reference counterpart: torch leaves its intermediates to the cache
 * (pro_b_gan_infer.py:201, :207). */
int pbg_set_workspace_discard(pbg_ctx* ctx, int on);

/* Result mirrors -- the output exchange of a batch-sharded multi-GPU job without a collective.  After this call every
 * bf16-mode pass of the ctx writes each result row not only to the caller's own gen_out / gen_scores / logits /
 * probs but also, at the same row index, to the n (<= 7) mirror buffers given here: device pointers into peer GPUs'
 * memory (peer access enabled: CUDA IPC, cuMem fabric handles, torch symmetric memory ...), already offset to the
 * caller's shard.  The stores travel over NVLink from the last layers' epilogues; they are complete when the pass
 * has completed on its stream, so readers on other GPUs need their usual cross-rank synchronisation (a barrier, a
 * flag) and nothing else.  An array may be NULL when the matching result is not requested; n = 0 clears.
 * Passes that cannot honour mirrors (fp32 mode, models too wide for the pair kernel) fail with PBG_ERR_UNSUPPORTED. */
int pbg_set_result_mirrors(pbg_ctx* ctx, int n, void* const* gen_out, float* const* gen_scores,
                           float* const* logits, float* const* probs);

/* Result multicast -- the same exchange through ONE store per 16 bytes instead of one per peer.  The four pointers are
 * NVSwitch multicast addresses (cuMulticast* objects; torch symmetric memory: handle.multicast_ptr) of symmetric result
 * buffers, already offset to the caller's shard; a NULL pointer leaves that result out; all NULL clears.  Every bf16-mode
 * pass then ALSO writes each result row with multimem.st to the multicast address, and the switch replicates the store
 * into every GPU's copy of the buffer (the caller's own copy included): NVLink egress per GPU is one copy of its
 * rows whatever the number of GPUs.  Completion and reader synchronisation as for mirrors.  The addresses must really
 * be multicast mappings: multimem.st to ordinary memory faults. */
int pbg_set_result_multicast(pbg_ctx* ctx, void* gen_out_mc, float* gen_scores_mc, float* logits_mc, float* probs_mc);

/* Entity scoring + top-k: the tail of ProtBGANInference.predict_tails (pro_b_gan_infer.py:146-151) and all of
 * find_similar_entities (:231-236):
 *     similarities = F.normalize(queries, dim=-1) @ F.normalize(table, dim=-1).T      [B, N], never materialised
 *     top_scores, top_indices = similarities.topk(k, dim=1)                           (largest first)
 * pbg_topk_prepare reads the fp32 table [N, E] once (row norms + a normalised bf16 copy; the reference re-normalises
 * all N rows on every call) -- call it again whenever the table changes.  pbg_topk scores fp32 queries [B, E] against
 * the prepared table.  E == 128, k <= 64 and N >= max(4096, 64 k x the sampling stride: 4 for k <= 16, 2 above): bf16 tensor-core scores of a table sample give a cut-off per row, a second
 * tensor-core pass over the whole table marks every entity above it, every marked entity is re-scored exactly in fp32
 * and a row whose k-th exact score does not provably beat everything that was not marked is redone by an exact scan.
 * Other shapes (k up to 512, any E): exact fp32 scores by a SIMT GEMM over chunks of rows + one selection CTA per row
 * (histogram of the row's scores, collect what lies at or above the k-th best's bin, sort).
 * Either way indices / scores are those of an fp32 evaluation (ties between equal scores: lower index first).
 * out_idx int64 [B, k], out_scores fp32 [B, k]; 1 <= k <= min(N, 512) (larger k: PBG_ERR_UNSUPPORTED).  Stream-ordered. */
int pbg_topk_prepare(pbg_ctx* ctx, const float* table, int64_t N, void* stream);
int pbg_topk(pbg_ctx* ctx, const float* queries, int64_t B, int k, int64_t* out_idx, float* out_scores, void* stream);
/* Diagnostics: how many query rows of the last pbg_topk chunk (<= 16384 rows) the tensor-core filter could not prove
 * and handed to the exact scan (0 when the general path ran).  Synchronises `stream`; -1 on error. */
int64_t pbg_topk_last_flagged(pbg_ctx* ctx, void* stream);

/* Host-side ingest of the CLI's index arrays; replaces json.loads (pro_b_gan_infer.py:485 --input_pairs, :493
 * --input_triplets, :501 --input_entities) + torch.tensor(list) (:135-136, :182, :226).  `text[0..len)` is the JSON
 * text: "[a, b, ...]" for cols == 1, "[[a, b], ...]" / "[[h, r, t], ...]" for cols == 2 / 3 (1 <= cols <= 8).  Ids are
 * JSON integers that fit int64; a float, a ragged row or any other token is PBG_ERR_INVALID with the byte offset in
 * pbg_last_error(NULL).  Writes at most cap_rows rows of `cols` int64 to `out` (out may be NULL to count) and
 * returns the number of rows in the text (>= 0), or -PBG_ERR_INVALID.  No ctx, no device, thread-safe. */
int64_t pbg_parse_index_rows(const char* text, size_t len, int cols, int64_t* out, size_t cap_rows);

/* Host-side result formatting; replaces `.tolist()` (pro_b_gan_infer.py:154, :162, :203, :208-209) + the list part of
 * json.dump(results, indent=2) (:503-508).  Writes the JSON text of a [rows, cols] array (cols == 0: a flat list of
 * `rows` scalars) exactly as json.dumps prints the corresponding Python list: fp32 values as the repr of the double
 * they convert to (shortest round-trip digits; NaN / Infinity like json.dumps), one item per line indented by
 * `indent` spaces per level with the array at nesting depth `depth`; indent < 0 gives the compact ", " form.
 * Returns the number of bytes the text needs (no terminator); nothing beyond `cap` bytes is written, so call with
 * out = NULL to size the buffer.  No ctx, no device, thread-safe. */
int64_t pbg_format_f32_json(const float* v, size_t rows, int cols, int indent, int depth, char* out, size_t cap);
int64_t pbg_format_i64_json(const int64_t* v, size_t rows, int cols, int indent, int depth, char* out, size_t cap);

/* Number of kernels this ctx has launched since creation (bench.py's gpu_launches). */
int64_t pbg_launch_count(const pbg_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* PBG_H_ */
