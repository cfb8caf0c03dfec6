/* b200rwkv.h — C ABI of the B200-native RWKV inference engine.
 *
 * This is the drop-in boundary underneath crates/ai00-core: every entry point replaces one
 * use of the `web-rwkv` crate at a call site of the reference (paths relative to the
 * reference repository root).  The Rust shim that implements web-rwkv's `Runtime<Rnn>` /
 * `State` traits on top of these functions is given in INTEGRATION.md.
 *
 * Conventions
 *   - every function returns 0 on success, a negative b200rwkv_status on failure; the message
 *     of the calling thread's most recent failure is available from b200rwkv_last_error()
 *     (thread-local: the infer task and the softmax task never see each other's text).  No
 *     exception crosses the boundary.
 *   - all buffers are caller-owned plain host memory unless stated; nothing is retained after
 *     the call returns (the `.st` image is only borrowed during b200rwkv_create).
 *   - threading mirrors the reference: ONE task calls infer/state ops
 *     (crates/ai00-core/src/run.rs:1232) and ONE task calls softmax (run.rs:1237); the engine
 *     serialises each group with an internal mutex.
 *   - there is no CPU fallback: creation fails if no sm_100 device is present.
 */
#ifndef B200RWKV_H
#define B200RWKV_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct b200rwkv_engine b200rwkv_engine;

typedef enum {
    B200RWKV_OK = 0,
    B200RWKV_ERR_INVALID = -1,     /* bad argument / malformed .st */
    B200RWKV_ERR_UNSUPPORTED = -2, /* model version or precision not supported */
    B200RWKV_ERR_CUDA = -3,        /* CUDA failure: the engine is dead, reload it */
    B200RWKV_ERR_STATE = -4        /* unknown slot / snapshot id */
} b200rwkv_status;

/* Mirror of web-rwkv `ModelInfo` as consumed at crates/ai00-core/src/lib.rs:587 and
 * crates/ai00-core/src/run.rs:672 (fields `version`, `num_vocab` are read by the core). */
typedef struct {
    int32_t version;            /* 5, 6 or 7 */
    int32_t num_layer;
    int32_t num_emb;
    int32_t num_hidden;
    int32_t num_vocab;
    int32_t num_head;
    int32_t head_size;
    int32_t time_mix_adapter;   /* v6 ddlerp LoRA rank */
    int32_t time_decay_adapter; /* v6 decay / v7 w LoRA rank */
} b200rwkv_info;

/* RnnOption (crates/ai00-core/src/run.rs:25, used at run.rs:710-724, 812-822). */
enum {
    B200RWKV_OPTION_LAST = 0,
    B200RWKV_OPTION_FULL = 1,
    /* consume the tokens, emit no logits: what a shim passes for a Last slot whose token run is
     * cut by token_chunk_size and continues in the next infer call (run.rs:1134-1145) */
    B200RWKV_OPTION_NONE = 2
};
/* Scoring options, accepted by b200rwkv_infer_score only (b200rwkv_infer answers B200RWKV_ERR_INVALID). */
#define B200RWKV_OPTION_SCORE 3
#define B200RWKV_OPTION_SCORE_KEPT 4

/* Replaces `Loader::info(&SafeTensors)` — crates/ai00-core/src/lib.rs:587,
 * crates/ai00-server/src/api/file.rs:115.  Pure host code, no GPU needed. */
int32_t b200rwkv_info_from_st(const uint8_t* st, size_t len, b200rwkv_info* out);

/* Replaces `ModelBuilder::new(ctx, st).build_vN()` + `vN::Bundle::<f16>::new(model, max_batch)`
 * + `TokioRuntime::<Rnn>::new(bundle)` — crates/ai00-core/src/lib.rs:484-515.
 * `device` is the CUDA ordinal (the reference's adapter selection, lib.rs:351-368).
 * precision (the reference's `Precision`, lib.rs:493: `Bundle::<f16>` / `Bundle::<f32>` = the ACTIVATION type; weights
 * are f16 on disk and in HBM either way):
 *   0 = fp16: every projection input is rounded to f16 (tensor-core operand), f32 accumulate / state / logits;
 *   1 = fp32: no activation is rounded -- every projection input travels as an f16 hi + lo pair (two operand tiles,
 *       accumulators added), which is f32-exact to ~2^-22; steps are capped at 16 tokens. */
int32_t b200rwkv_create(const uint8_t* st, size_t len, int32_t device, int32_t max_batch,
                        int32_t token_chunk_size, int32_t precision, b200rwkv_engine** out);

/* Everything the reference's ReloadRequest carries for this path (crates/ai00-core/src/lib.rs:196-240, 484-497), one call:
 *   - devices: `num_devices` in {1, 2, 4, 8} CUDA ordinals of this box.  With more than one, the returned handle is ONE engine
 *     that owns every tensor-parallel rank (head / column parallel, SURVEY.md §8e) and one worker thread per rank: every call
 *     below is made once, by the same two tasks as before, and drives all GPUs -- the reference's single `Runtime` object
 *     (run.rs:1230-1234).  State tensors are merged / scattered by head inside state_back / state_load.
 *   - LoRA files blended into the projection matrices while they are uploaded (lib.rs:466-485, `LoraBlend::full(alpha)`):
 *     `<name>.lora.1` [out, r] and `<name>.lora.0` [in, r] as the reference's converter writes them
 *     (assets/scripts/convert_safetensors.py:96-101); W += alpha * lora.1 @ lora.0^T in f32, rounded once to f16.  Files with
 *     anything but low-rank pairs on att.{receptance,key,value,gate,output} / ffn.{key,value,receptance} / head are
 *     B200RWKV_ERR_UNSUPPORTED.  Images are borrowed during the call only.
 * Set struct_bytes = sizeof(b200rwkv_options); zero the rest for defaults (device 0, no LoRA, fp16). */
#define B200RWKV_MAX_LORA 4
typedef struct {
    uint32_t struct_bytes;
    int32_t max_batch, token_chunk_size, precision;
    int32_t num_devices;              /* 0 or 1: single GPU, devices[0] (0 if num_devices == 0) */
    int32_t devices[8];
    int32_t num_lora;
    const uint8_t* lora_st[B200RWKV_MAX_LORA];
    size_t lora_len[B200RWKV_MAX_LORA];
    float lora_alpha[B200RWKV_MAX_LORA];
    /* `quant` / `quant_type` of the reload request (lib.rs:211-215, 465: the first `quant_layers` layers keep their eight
     * projection matrices in a weight-only quantised format; everything else stays f16).  Single GPU, precision 0 only. */
    int32_t quant_layers;
    int32_t quant_type;               /* B200RWKV_QUANT_* */
} b200rwkv_options;
#define B200RWKV_QUANT_NONE 0
#define B200RWKV_QUANT_INT8 1         /* blocks of 128 inputs: f16 (min, max) + 8-bit codes */
#define B200RWKV_QUANT_NF4 2          /* blocks of 64 inputs: f16 absmax + 4-bit NormalFloat codes */
                                      /* Quant::SF4 is not implemented: create_ex answers B200RWKV_ERR_UNSUPPORTED */
int32_t b200rwkv_create_ex(const uint8_t* st, size_t len, const b200rwkv_options* opt, b200rwkv_engine** out);

/* Tensor-parallel construction, one process per GPU (head / column parallel, SURVEY.md §8e).
 * (The in-process alternative -- one handle, all ranks inside -- is b200rwkv_create_ex above.)
 * Every rank calls create_tp with the same model, then exchanges the opaque handle blobs
 * (b200rwkv_tp_export on each rank, all-gathered by the host over any side channel) and
 * passes all `world` blobs, rank-ordered, to b200rwkv_tp_connect.  After that every API call
 * is SPMD: all ranks make the same call with the same arguments.  Rank 0 receives the full
 * [rows, num_vocab] logits (gathered from every rank's vocabulary shard over NVLink peer
 * memory); the other ranks' logits_out may be NULL.  State tensors are sharded by head:
 * state_back on rank r fills the WKV rows of its own heads and zeros elsewhere. */
#define B200RWKV_TP_HANDLE_BYTES 128
int32_t b200rwkv_create_tp(const uint8_t* st, size_t len, int32_t device, int32_t max_batch,
                           int32_t token_chunk_size, int32_t precision, int32_t rank, int32_t world,
                           b200rwkv_engine** out);
int32_t b200rwkv_tp_export(b200rwkv_engine*, uint8_t handle_out[B200RWKV_TP_HANDLE_BYTES]);
int32_t b200rwkv_tp_connect(b200rwkv_engine*, const uint8_t* handles /* world * HANDLE_BYTES */);
/* Same wiring when all ranks live in one process (rank-ordered array of engines). */
int32_t b200rwkv_tp_connect_local(b200rwkv_engine** engines, int32_t n);

/* Dropping the `Arc<dyn Runtime>` (crates/ai00-core/src/lib.rs:600,654). */
void b200rwkv_destroy(b200rwkv_engine*);

int32_t b200rwkv_get_info(b200rwkv_engine*, b200rwkv_info* out);

/* Replaces `Runtime::infer(RnnInput)` — crates/ai00-core/src/run.rs:1143 — for one
 * `RnnInput`: a ragged batch of `nslot` entries; entry i feeds `ntok[i]` tokens
 * (tokens + sum(ntok[0..i])) to state slot `slot[i]` with RnnOption `option[i]`.
 * All tokens are consumed (internally in steps of at most min(token_chunk_size, 128) tokens shared evenly over the
 * entries, the policy
 * web-rwkv applies across calls at run.rs:1134-1145).  Logits rows (num_vocab f32 each) are
 * written contiguously to `logits_out` in entry order: 1 row for LAST (0 if ntok[i]==0),
 * ntok[i] rows for FULL, none for NONE; rows_out[i] receives the row count of entry i
 * (== RnnOutputBatch being empty or not, run.rs:1146-1155).  `logits_cap` is in floats.
 * `logits_out` may be NULL: nothing is copied to the host, the last row of every slot stays in HBM for
 * b200rwkv_sample_topk.  Token ids >= num_vocab are B200RWKV_ERR_INVALID. */
int32_t b200rwkv_infer(b200rwkv_engine*, int32_t nslot, const int32_t* slot, const int32_t* ntok,
                       const uint32_t* tokens, const int32_t* option, float* logits_out,
                       size_t logits_cap, int32_t* rows_out);

/* Replaces the forward pass of the reference's perplexity() -- crates/ai00-core/src/run.rs:699-755, run once per choice (twice
 * with `calibrate`) by the chooses endpoint, run.rs:936-983 -- which copies one num_vocab f32 row per token to the host and
 * normalises it there to read one number.  Same arguments and results as b200rwkv_infer, and additionally:
 * an entry with option SCORE or SCORE_KEPT holding tokens x0 .. x{n-1} steps like FULL but copies no logits rows
 * (rows_out[i] = 0); its last row becomes the slot's kept row, as for LAST with logits_out = NULL.  It writes n floats to
 * `logp_out`, packed in entry order over the scoring entries only:
 *     logp[j] = log_softmax(row of x{j-1})[x{j}]          j >= 1
 *     logp[0] = NaN                                        SCORE
 *     logp[0] = log_softmax(kept row at call start)[x0]    SCORE_KEPT (the reference's `head` term; chained calls are exact)
 * `logp_cap` is in floats.  Refused before any step runs, so a refused call changes no state:
 *     SCORE_KEPT on a slot with no kept row                             B200RWKV_ERR_STATE
 *     logp_out == NULL with scoring entries, or logp_cap too small      B200RWKV_ERR_INVALID
 *     SCORE_KEPT where the engine keeps no rows (num_vocab / world % 4) B200RWKV_ERR_UNSUPPORTED
 * Tensor parallel (create_tp): SPMD like b200rwkv_infer; rank 0 fills logp_out, the other ranks may pass NULL. */
int32_t b200rwkv_infer_score(b200rwkv_engine*, int32_t nslot, const int32_t* slot, const int32_t* ntok,
                             const uint32_t* tokens, const int32_t* option, float* logits_out, size_t logits_cap,
                             int32_t* rows_out, float* logp_out, size_t logp_cap);

/* `State` trait object — crates/ai00-core/src/lib.rs:399,494; uses at run.rs:477,1099-1107.
 * The host-visible state of one slot is an f32 tensor of web-rwkv shape [C, N+2, L, 1]
 * (x fastest; run.rs:987): row 0 time-mix shift, rows 1..N WKV, row N+1 channel-mix shift. */
int32_t b200rwkv_state_shape(b200rwkv_engine*, int64_t shape[4]);
int32_t b200rwkv_state_init(b200rwkv_engine*, float* out);                          /* State::init  */
int32_t b200rwkv_state_load(b200rwkv_engine*, int32_t slot, const float* in);        /* State::load  */
int32_t b200rwkv_state_back(b200rwkv_engine*, int32_t slot, float* out);             /* State::back  */
int32_t b200rwkv_state_read(b200rwkv_engine*, int32_t slot, uint64_t* snapshot_id);  /* State::read  (device copy) */
int32_t b200rwkv_state_write(b200rwkv_engine*, int32_t slot, uint64_t snapshot_id);  /* State::write */
int32_t b200rwkv_state_free(b200rwkv_engine*, uint64_t snapshot_id);                 /* drop TensorGpu */

/* Device-resident state cache (SURVEY.md §8f-4).  The reference's cache holds `CachedItem { state: TensorCpu, output:
 * TensorCpu }` (crates/ai00-core/src/run.rs:199-205): every check-out / check-in is a State::load / State::back PCIe copy of
 * the whole state (34.6 MB per slot at 7B; run.rs:838, 996, 561).  Here a cached item is a snapshot id: state_read /
 * state_write are device-to-device copies, and the snapshot carries the slot's last logits row with it, so a cache hit can
 * be sampled on the device (b200rwkv_sample_topk) without re-running a token.  The two calls below move a snapshot to / from
 * host tensors without occupying a slot -- for spilling under memory pressure (b200rwkv_cache_stats), for `InputState::Value`
 * / `.state` files (run.rs:390-437) and for `/api/oai/states` (run.rs:984-989).  state: [C, N+2, L, 1] f32 as in
 * b200rwkv_state_back; logits: [num_vocab] f32, either pointer may be NULL (logits_out: ERR_STATE if the snapshot has no row). */
int32_t b200rwkv_snapshot_back(b200rwkv_engine*, uint64_t snapshot_id, float* state_out, float* logits_out);
int32_t b200rwkv_snapshot_load(b200rwkv_engine*, const float* state_in, const float* logits_in, uint64_t* snapshot_id);
int32_t b200rwkv_cache_stats(b200rwkv_engine*, int64_t* num_snapshots, int64_t* bytes_used, int64_t* bytes_free);

/* Replaces `vN::read_state(&context, &info, reader)` — crates/ai00-core/src/lib.rs:378-389 (initial states of state-tuned
 * models and `.state` files, run.rs:403-437): reads `blocks.{l}.att.time_state` [H, N, N] (F16 / F32 / BF16; the layout the
 * converter writes, crates/converter/src/main.rs:20) into the state tensor `out` ([C, N+2, L, 1] f32).  Host only. */
int32_t b200rwkv_read_state(const b200rwkv_info* info, const uint8_t* st, size_t len, float* out);

/* Replaces `web_rwkv::runtime::softmax::softmax(&context, Vec<TensorCpu<f32>>)` —
 * crates/ai00-core/src/run.rs:1179.  in/out: [rows, num_vocab] f32. */
int32_t b200rwkv_softmax(b200rwkv_engine*, int32_t rows, const float* in, float* out);

/* GPU front half of token sampling (SURVEY.md §8f-1).  Replaces, for samplers that only need the head of the sorted
 * distribution (Nucleus with top_k <= 128 -- the reference default, sampler/nucleus.rs:16-17 -- and greedy), the per-token
 * per-slot sequence of crates/ai00-core/src/run.rs:664-697: `output.to_vec()` (num_vocab f32 D2H), `Sampler::transform`
 * (penalties, sampler/nucleus.rs:61-67), `Formatter::transform` (BNF mask, sampler/bnf.rs:37-40), the bias add
 * (run.rs:679-681), the softmax round trip (run.rs:1164-1190) and the full-vocabulary sort of
 * sampler/nucleus.rs:69-80.  Pass `logits_out = NULL` to b200rwkv_infer: the logits stay in HBM, and this call returns, for
 * each listed slot, the `top_k` most probable tokens of that slot's most recent logits row after
 *     logits[penalty_token[j]] -= penalty_value[j]     j in [penalty_offset[i], penalty_offset[i+1])
 *     logits[t] = -inf  where bit t of allow_bits row i is 0                    (allow_bits may be NULL)
 *     logits[bias_token[j]]    += bias_value[j]        j in [bias_offset[i], bias_offset[i+1])
 * (tokens distinct within one row's penalty list and within its bias list, as the reference's HashMaps are), with
 * probs = softmax over the whole adjusted row.  Order: logit descending, token id ascending on ties.  ids_out / probs_out:
 * [nrows][top_k].  The draw itself (top_p cut, temperature, RNG, penalty update; nucleus.rs:81-123) stays in the host
 * sampler, now over <= 128 pairs.  Samplers that need the whole distribution (Mirostat, Typical) keep using
 * b200rwkv_infer with a logits buffer + b200rwkv_softmax.  Thread contract: the softmax task's (run.rs:1237). */
int32_t b200rwkv_sample_topk(b200rwkv_engine*, int32_t nrows, const int32_t* slots, const int32_t* penalty_offset,
                             const uint32_t* penalty_token, const float* penalty_value, const uint32_t* allow_bits,
                             const int32_t* bias_offset, const uint32_t* bias_token, const float* bias_value, int32_t top_k,
                             uint32_t* ids_out, float* probs_out);

/* Pinned host memory for logits / state buffers (full-rate DMA); optional. */
int32_t b200rwkv_host_alloc(size_t bytes, void** out);
void b200rwkv_host_free(void* p);

/* Measurement hook used by bench.py for the kernel-resident number: runs `warmup + steps`
 * decode steps (one token per listed slot per step) with token ids staged in HBM beforehand,
 * no host<->device traffic inside the timed region; returns CUDA-event milliseconds for the
 * `steps` timed steps and the number of kernel launches in that region.  The last logits row of
 * every listed slot stays in HBM as after b200rwkv_infer with logits_out = NULL. */
int32_t b200rwkv_bench_decode(b200rwkv_engine*, int32_t nslot, const int32_t* slot,
                              const uint32_t* tokens /* [(warmup+steps) * nslot] */, int32_t warmup,
                              int32_t steps, int32_t flush_l2, float* ms_out, int64_t* launches_out,
                              float* step_ms_out /* optional [steps]: CUDA-event time of every timed step */);

/* Per-kernel-class device time of ONE un-graphed decode step, CUDA events around every launch
 * on the engine's stream.  classes: 0 = projection GEMMs, 1 = WKV, 2 = LN/mix/embed, 3 = other.
 * ms[4], launches[4], and algorithmic weight bytes streamed by the GEMM launches. */
int32_t b200rwkv_profile_step(b200rwkv_engine*, int32_t nslot, const int32_t* slot,
                              const uint32_t* tokens, float ms[4], int32_t launches[4],
                              int64_t* gemm_weight_bytes);

/* In-situ per-launch windows of ONE graph-replayed decode step (globaltimer stamps written by the kernels themselves):
 * window = [griddepcontrol.wait released, last CTA exit]; consecutive windows cannot overlap, so class sums are <= the step.
 * types[i]: 0 LN / mix, 2 WKV, 6 fused RWKV-6 front half, 1000000 + weight MiB for a projection launch; bytes[i]: algorithmic
 * weight bytes of a projection launch (else 0); start_us / end_us relative to the first stamp of the step, averaged over
 * `reps` replays; step_us = last exit - first entry.  bench.py's `roofline` comes from here. */
int32_t b200rwkv_profile_insitu(b200rwkv_engine*, int32_t nslot, const int32_t* slot, const uint32_t* tokens, int32_t reps,
                                int32_t cap, int32_t* n_out, int32_t* types, double* start_us, double* end_us, int64_t* bytes,
                                double* step_us);

/* Operator-level entry (parity tests): one launch of the WKV kernel -- recurrence + per-head GroupNorm (eps 64e-5) (+ v7
 * bonus) * gate -- on caller-supplied head vectors, for one sequence of T <= 64 tokens with H heads of size 64; no model.
 * r, k, v, g: [T, H*64] (g NULL = 1); w: decay in (0, 1), [T, H*64] (v5: static [H*64]); u: v5/v6 time_first [H*64];
 * v7: a [T, H*64], k_k / k_a / r_k [H*64] (kk = normalize_head(k * k_k), k <- k * (1 + (a - 1) * k_a), value-residual off);
 * lnx_w / lnx_b [H*64] (NULL = 1 / 0); state: in/out [H][64][64] in the device orientation M[value][key] (v5/v6: the
 * transpose of S[key][value]); out: [T, H*64], the f16 values the kernel hands to the output projection.  The committed
 * flash-linear-attention fixtures (tests/golden/wkv6_fla.npz, wkv7_fla.npz) are checked through this entry. */
/* Operator-level entry (parity tests): the load-time quantiser on a caller-supplied row-major f16 matrix [N, K] (K % 128 == 0),
 * returned in plain order: codes [N, K] (one byte per element: Int8 code, or NF4 level index 0..15), p0 [N, K/block] (Int8: block
 * minimum, NF4: block absmax), p1 [N, K/block] (Int8: the scale f16((max - min) / 255); NF4: unused, may be NULL).  p0 / p1 are f16
 * bit patterns.  block = 128 (Int8) or 64 (NF4). */
int32_t b200rwkv_op_quantize(int32_t device, int32_t quant_type, int32_t N, int32_t K, const uint16_t* w_f16, uint8_t* codes,
                             uint16_t* p0, uint16_t* p1);

int32_t b200rwkv_op_wkv(int32_t device, int32_t version, int32_t T, int32_t H, const float* r, const float* k, const float* v,
                        const float* w, const float* u, const float* a, const float* k_k, const float* k_a, const float* r_k,
                        const float* g, const float* lnx_w, const float* lnx_b, float* state, float* out);

/* Kernels launched by this engine's forward steps since creation (graph replays counted by their kernel nodes). */
int32_t b200rwkv_launch_count(b200rwkv_engine*, int64_t* total);

/* The residual stream after the last layer, one [num_emb] f32 row per token -- the hidden state the documented embeddings
 * route returns (reference docs/doc-api/openai.md:376-437).  After b200rwkv_keep_hidden(e, 1) every infer call records the
 * rows of ALL its tokens (entry order, like the token array); without it only the rows of the call's last internal step
 * (<= 128 tokens) are available.  b200rwkv_last_hidden returns the number of rows written (negative status on error). */
int32_t b200rwkv_keep_hidden(b200rwkv_engine*, int32_t enable);
int32_t b200rwkv_last_hidden(b200rwkv_engine*, float* out, size_t cap);

/* Test aid: copy a named internal activation buffer of the most recent internal step of b200rwkv_infer to the host as f32
 * row-major [*rows_out, cols]; returns the column count (negative status on error).  rows = the step's tokens, or its output
 * rows for the head's operand "a_head".  A16 operands of a split-operand step (precision 1) are returned as hi + lo.  Not on
 * the product path. */
int32_t b200rwkv_debug_read(b200rwkv_engine*, const char* name, float* out, size_t cap, int32_t* rows_out);

/* Test aid: the projection launches a step of `mt` token tiles (1, 2, 4, 8) runs for layer `layer` (-1 = the head, at `mt`
 * output-row tiles), in stream order.  One record of B200RWKV_PLAN_INTS int32 per launch:
 *   [0] grid the step launches  [1] grid  [2] grid_wide  [3] total_blocks  [4] max_contrib  [5] qtype (0 f16, 1 Int8, 2 NF4)
 *   [6] 1 = grid fixed by a static split-K  [7] nseg, then per segment (up to 8) five ints: KB, tiles, N, out_mode, act.
 * CTA c of a launch streams the 128 x 128 blocks [c * total_blocks / grid, (c + 1) * total_blocks / grid) of the launch's
 * segments in order (tile-major, k blocks within a tile).  Returns the number of launches (negative status on error). */
#define B200RWKV_PLAN_INTS 48
int32_t b200rwkv_debug_plan(b200rwkv_engine*, int32_t layer, int32_t mt, int32_t* out, size_t cap);

/* Profiling aid: raw stamp rows of the most recent b200rwkv_profile_insitu replay, one row of 512 uint64 per launch
 * (out = [launches][512]): globaltimer stamps of CTA 0 in [0..7] (entry, past griddepcontrol.wait, phase marks, exit), then
 * {SM id, last MMA issued, exit} of every projection CTA (or {entry, released, phase 1 done} of every CTA of the fused RWKV-6
 * front-half kernel); types[i] = 0 LN, 2 WKV, 6 front half, 1000000 + weight MiB for a projection launch. */
int32_t b200rwkv_debug_trace(b200rwkv_engine*, uint64_t* out, size_t cap, int32_t* types, int32_t* nphase);

/* Profiling aid: one projection launch class timed in isolation over all layers. */
int32_t b200rwkv_debug_gemm_time(b200rwkv_engine*, int32_t which, int32_t reps, float* ms_out, int64_t* bytes_out,
                                 uint64_t* trace_out);

#ifdef B200RWKV_DEBUG
/* Debug build only (libb200rwkv_dbg.so, `python -m ai00_server_b200.build --debug`): HBM streaming and L2 prefetch
 * micro-benchmarks (csrc/streamtest.cuh).  The debug build also honours the B200RWKV_* bring-up environment switches;
 * the product library ignores the environment. */
int32_t b200rwkv_debug_stream(int32_t device, int32_t kind, double gbytes, int32_t stage_bytes, int32_t nstage,
                              int32_t use_hint, int32_t consumer, int32_t split, int32_t producers, int32_t reps,
                              float* ms_out);
int32_t b200rwkv_debug_prefetch(int32_t device, double mbytes, int32_t consumers, int32_t pf_grid, int32_t skip, int32_t nblk,
                                int32_t mode, double idle_us, int32_t reps, float* ms_out);
/* SM cycles for n back-to-back tcgen05.mma kind::f16 of shape [M x 16] x [16 x N] on one SM, A operand from shared memory or
 * tensor memory: cycles[0] = the issue loop, cycles[1] = until the last one has retired. */
int32_t b200rwkv_debug_mma_rate(int32_t device, int32_t M, int32_t N, int32_t a_in_tmem, int32_t n, int64_t* cycles);
#endif

const char* b200rwkv_last_error(b200rwkv_engine*);

#ifdef __cplusplus
}
#endif
#endif /* B200RWKV_H */
