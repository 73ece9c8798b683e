/* libcvk - C ABI of the B200-native CosyVoice2 hot path (LM decode -> CFM flow -> HiFT vocoder + mel frontend).
 *
 * This header is the drop-in boundary (SURVEY.md §8b).  The reference is pure Python, so there is no FFI to
 * mirror symbol-for-symbol; each entry point replaces one of the engine plug-in granularities the reference itself
 * swaps (TensorRT estimator, vLLM LM, TorchScript encoder) or one stage-model method, cited per function as
 * "replaces <file>:<lines>" relative to the reference tree.
 *
 * Conventions
 *  - Every pointer is a DEVICE pointer unless its name ends in _host.  Memory is owned by the caller (PyTorch
 *    allocates it); the library owns only its repacked weights, KV arena and workspace, all inside cvk_ctx.
 *  - Activations cross the ABI as *ragged time-major* fp32 matrices: the B sequences are concatenated along
 *    rows without padding, `lens_host[b]` rows each, channels contiguous ([sum(lens), C]).
 *  - Every data-path call takes an explicit cudaStream_t (passed as void*), never touches the default stream on its own
 *    and never calls cudaDeviceSynchronize (set-up calls - cvk_create / cvk_set_tensor / cvk_finalize / cvk_profile /
 *    cvk_destroy - repack weights on the default stream and block until done).
 *  - Threading: calls that use the ctx workspace (cvk_lm_prefill, cvk_lm_forward_logp, every flow / vocoder / mel / op
 *    call) must be serialised by the caller.  Calls that only touch an LM session (cvk_lm_decode, cvk_lm_begin,
 *    cvk_lm_feed, cvk_lm_next_logp, cvk_lm_last_logits) and cvk_ras_sample own no shared state: they may run
 *    concurrently with workspace calls and with each other on DISTINCT sessions and streams - this is the reference's
 *    own concurrency (LM side thread + side stream next to token2wav, cli/model.py:101-129, 268; several requests in
 *    flight, runtime/python/grpc/server.py:69).  One session is never used by two host threads at once.  Streaming-flow
 *    sessions (cvk_flow_stream_*, one slot or several) hold caches only: their begin / chunk / chunk_batch calls use the
 *    workspace and are serialised like every other flow call.
 *  - Return value: 0 on success, a negative cvk_status otherwise; cvk_last_error(ctx) holds the message.  No C++
 *    exception crosses the ABI.  There is NO CPU fallback: without a CUDA device cvk_create fails.
 */
#ifndef CVK_H_
#define CVK_H_
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cvk_ctx cvk_ctx;

typedef enum {
  CVK_OK = 0,
  CVK_ERR_INVALID = -1,        /* bad argument / shape (reference: AssertionError / ValueError) */
  CVK_ERR_CUDA = -2,           /* CUDA runtime / driver error */
  CVK_ERR_OOM = -3,            /* workspace or KV arena exhausted */
  CVK_ERR_MISSING_WEIGHT = -4, /* a state_dict key required by cvk_finalize was not supplied */
  CVK_ERR_STATE = -5           /* stage not finalised / session misuse */
} cvk_status;

/* arithmetic of the tensor-core stages */
#define CVK_PREC_FP32 0 /* everything fp32 on CUDA cores: parity mode, tracks the CPU reference to ~1e-4 */
#define CVK_PREC_BF16 1 /* dense GEMM / conv operands bf16 on tcgen05 tensor cores, fp32 accumulate + residuals */

/* ---------------------------------------------------------------------------------------------- context */
int cvk_create(int device, int precision, size_t workspace_bytes, cvk_ctx** out);
void cvk_destroy(cvk_ctx* ctx);
const char* cvk_last_error(cvk_ctx* ctx);
const char* cvk_version(void);
/* kernels launched by this library since creation (bench.py "gpu_launches") */
int64_t cvk_launch_count(cvk_ctx* ctx);
/* mean device time (ms) of the kernel timed by the last cvk_op_* call when the "op_iters" option is > 0 (tools/gemm_probe.py) */
double cvk_last_op_ms(cvk_ctx* ctx);
/* debug: copy (and clear) the device timeline buffer filled by instrumented kernels when "debug_timeline" is on */
int cvk_debug_read(cvk_ctx* ctx, long long* out, int n);
/* workspace arena of the context (SURVEY.md §8b `cvk_workspace_bytes`): capacity given to cvk_create and the high-water mark of
 * the calls made so far - what a caller needs to size cvk_create for its largest batch. */
int cvk_workspace_bytes(cvk_ctx* ctx, size_t* capacity, size_t* high_water);
/* Test / measurement switches, NOT part of the drop-in surface (every default is the benchmarked configuration): kernel-variant
 * A/B ("use_tc", "tc_persist", "tc_bn256", "tc_pbn256", "tc_epi", "use_tc_attn", "attn_single_pass", "enc_tc_attn", "use_skinny",
 * "lm_fused", "lm_mega", "mega_coop", "pdl", "use_graph", "hift_f16" - the last one takes effect at the next cvk_finalize("hift")),
 * probes ("op_iters", "op_out_bf16", "debug_timeline", "chain_timeline").  Unknown keys return CVK_ERR_INVALID. */
int cvk_set_option(cvk_ctx* ctx, const char* key, int value);

/* Per-kernel-family device timing for the roofline report of bench.py: CUDA events are recorded around every launch
 * of a family while enabled (family 0 = tcgen05 conv-GEMM, 1 = CUDA-core conv-GEMM, 2 = attention).  Launches inside
 * the captured LM decode graph are not instrumented.  cvk_profile_read sums elapsed ms, algorithmic FLOPs and bytes. */
int cvk_profile(cvk_ctx* ctx, int enable);
int cvk_profile_read(cvk_ctx* ctx, int family, double* ms, double* flops, double* bytes, int64_t* launches);

/* ---------------------------------------------------------------------------------------------- weights
 * replaces cosyvoice/cli/model.py:65-73 (CosyVoice2Model.load -> load_state_dict(strict=True)).
 * `name` = "<stage>." + reference state_dict key, stage in {"llm","flow","hift"}; data fp32, C-contiguous, on the
 * device (on_device=1) or host.  cvk_finalize(stage) folds weight-norm (g*v/||v||), repacks convolutions to
 * [Cout][tap][Cin], builds polyphase transposed-conv weights and bf16 copies, then drops the raw tensors.
 * cfg: hift: none; flow: {enc_blocks, enc_up_blocks, num_mid_blocks, n_blocks}; llm: {num_layers}. */
int cvk_set_tensor(cvk_ctx* ctx, const char* name, const float* data, int on_device, const int64_t* shape, int ndim);
int cvk_finalize(cvk_ctx* ctx, const char* stage, const int* cfg, int ncfg);

/* ---------------------------------------------------------------------------------------------- generic ops
 * exposed for per-op parity tests (tests/test_ops_gpu.py); same kernels the stages use. */
/* out[r,n] = act(bias[n] + sum_j sum_k x[r + shift0 + j*dil, k] * w[n,k,j]) for one zero-padded sequence per
 * entry of lens_host.  w is a torch Conv1d weight [N,K,taps] fp32 on the device. */
int cvk_op_conv1d(cvk_ctx* ctx, const float* x, const int* lens_host, int B, int K, const float* w, const float* bias,
                  int N, int taps, int dil, int shift0, int act, float* out, void* stream);
/* out[b,n] = bias[n] + sum_k x[b,k] w[n,k] through the LM decode weight-streaming kernel (bf16 context, rows <= 64);
 * runs it `iters` more times and reports the mean device time; timeline_host (optional, 128 int64) receives the clock64
 * stamps of CTA 0 when the "debug_timeline" option is on. */
int cvk_op_linear_small(cvk_ctx* ctx, const float* x, int rows, int K, const float* w, const float* bias, int N, float* out, int iters,
                        float* ms_out, long long* timeline_host, void* stream);
/* block-causal / full multi-head attention over ragged sequences; q,k,v,out [sum(lens), H*64] */
int cvk_op_attention(cvk_ctx* ctx, const float* q, const float* k, const float* v, const int* lens_host, int B, int H,
                     int chunk, float scale, float* out, void* stream);

/* ---------------------------------------------------------------------------------------------- HiFT vocoder
 * replaces cosyvoice/hifigan/generator.py:557-569 (HiFTGenerator.inference) and its parts. */
/* f0_predictor.py:56-59: mel [sum T,80] -> f0 [sum T] */
int cvk_hift_f0(cvk_ctx* ctx, const float* mel, const int* lens_host, int B, float* f0, void* stream);
/* generator.py:560-564 + SourceModuleHnNSF/SineGen2: f0 [sum T], noise [sum 480T, 9] (standard-normal draws, the
 * reference's randn_like) -> source [sum 480T] */
int cvk_hift_source(cvk_ctx* ctx, const float* f0, const int* lens_host, int B, const float* noise, float* source,
                    void* stream);
/* generator.py:507-539 (decode): mel [sum T,80], source [sum 480T] -> wav [sum 480T] (clamped to +-0.99) */
int cvk_hift_decode(cvk_ctx* ctx, const float* mel, const int* lens_host, int B, const float* source, float* wav,
                    void* stream);
/* whole inference(); cache_source (optional, may be NULL) [sum cache_lens] overwrites the head of each source
 * (generator.py:566-567, streaming glue).  Outputs wav [sum 480T], source [sum 480T]. */
int cvk_hift_inference(cvk_ctx* ctx, const float* mel, const int* lens_host, int B, const float* noise,
                       const float* cache_source, const int* cache_lens_host, float* wav, float* source, void* stream);

/* ---------------------------------------------------------------------------------------------- flow (token -> mel)
 * replaces cosyvoice/flow/flow.py:235-281 (CausalMaskedDiffWithXvec.inference) and the engine plug-in points
 * flow/flow_matching.py:126-153 (forward_estimator: the TensorRT swap point) and cli/model.py:277-279 (encoder). */
/* transformer/upsample_encoder.py:244-307 on token ids.  tokens [sum N] int32 (prompt ++ generated per sequence).
 * context_len: 0 (finalize) or 3 (the last 3 tokens of every sequence are look-ahead context only,
 * flow.py:259-261).  out h [sum 2*(N-context_len), 512]. */
int cvk_flow_encoder(cvk_ctx* ctx, const int32_t* tokens, const int* lens_host, int B, int streaming, int context_len,
                     float* h, void* stream);
/* flow/decoder.py:405-494 (CausalConditionalDecoder.forward) - same I/O contract as the TensorRT engine:
 * x, mu, cond [sum T,80]; t [B]; spks [B,80]; out [sum T,80]; mask = ones within each length. */
int cvk_cfm_estimator(cvk_ctx* ctx, const float* x, const float* mu, const float* t, const float* spks, const float* cond,
                      const int* lens_host, int B, int streaming, float* out, void* stream);
/* the engine contract itself (flow/flow_matching.py:140-148: the last binding of the TensorRT context is x.data_ptr(), the
 * result overwrites x).  `out` of cvk_cfm_estimator may alias `x` as well: x is consumed before the first write. */
int cvk_cfm_estimator_inplace(cvk_ctx* ctx, float* x, const float* mu, const float* t, const float* spks, const float* cond,
                              const int* lens_host, int B, int streaming, void* stream);
/* flow/flow_matching.py:203-227 + 71-124: fixed seed-0 noise unless z given ([sum T,80]), cosine schedule, Euler,
 * CFG.  mu, cond [sum T,80]; spks [B,80]; out mel [sum T,80]. */
int cvk_cfm_solve(cvk_ctx* ctx, const float* mu, const float* spks, const float* cond, const int* lens_host, int B,
                  const float* z, int n_timesteps, float cfg_rate, int streaming, float* out, void* stream);
/* flow.py:235-281 end to end.  tokens [sum (P_b+N_b)] (prompt then generated), prompt_feat [sum Tp_b, 80],
 * embedding [B,192]; finalize=0 treats the last 3 tokens as look-ahead.  out mel [sum (2*(P+N-ctx) - Tp), 80]. */
int cvk_flow_inference(cvk_ctx* ctx, const int32_t* tokens, const int* token_lens_host, const float* prompt_feat,
                       const int* prompt_feat_lens_host, const float* embedding, int B, int n_timesteps, int streaming,
                       int finalize, float* mel, void* stream);

/* ---- incremental streaming flow (SURVEY 8(f) rank 1) -------------------------------------------------------------------------
 * The reference's streaming loop calls flow.inference(streaming=True, finalize=False) on the GROWING token prefix for every
 * chunk (cli/model.py:346-363) and keeps only the frames past token_offset.  Block-causal attention (utils/mask.py:127-158,
 * static chunk 50 frames) and causal convolutions (flow/decoder.py:25-62) make every complete chunk independent of later
 * frames, so a session object caches, per Euler step, the K/V rows of every estimator transformer block and the two-row
 * input tails of every causal convolution; a chunk call then computes its NEW frames only and returns exactly the rows the
 * reference call would (same noise rows of cvk_cfm_set_noise, same prompt conditioning).  Chunk ends must be multiples of
 * 50 frames (the reference's hop schedule guarantees it); the final, non-streaming call (finalize=True runs with
 * streaming=False in the reference, cli/model.py:372-378: full attention) stays cvk_flow_inference.
 * create: caches for up to max_frames mel frames (prompt included) and n_timesteps Euler steps; cvk_flow_stream_bytes reports
 * their size.  begin: new utterance - prompt_feat [prompt_frames,80], embedding [192] (device).  chunk: tokens = device
 * [n_tokens] prompt tokens + all speech tokens so far + the 3 look-ahead tokens; writes the frames
 * [max(done, prompt_frames), 2*(n_tokens-3)) to mel_out [mel_capacity_frames,80] and their count to *n_frames_out (host).
 * Calls on one session are serialised by the caller, like every workspace call of the context. */
typedef struct cvk_flow_stream cvk_flow_stream;
int cvk_flow_stream_create(cvk_ctx* ctx, int max_frames, int n_timesteps, cvk_flow_stream** out);
/* the same session for the CosyVoice3 DiT (stage "flow3", flow/flow.py:369-414 with streaming=True): K/V rows of the 22 blocks
 * (rotary positions absolute) and the 30-row input tails of the two grouped k31 position convolutions (DiT/modules.py:115-145);
 * begin / chunk / destroy / bytes are shared */
int cvk_flow3_stream_create(cvk_ctx* ctx, int max_frames, int n_timesteps, cvk_flow_stream** out);
void cvk_flow_stream_destroy(cvk_ctx* ctx, cvk_flow_stream* fs);
long long cvk_flow_stream_bytes(const cvk_flow_stream* fs);
int cvk_flow_stream_begin(cvk_ctx* ctx, cvk_flow_stream* fs, const float* prompt_feat, int prompt_frames, const float* embedding,
                          void* stream);
int cvk_flow_stream_chunk(cvk_ctx* ctx, cvk_flow_stream* fs, const int32_t* tokens, int n_tokens, float* mel_out,
                          int mel_capacity_frames, int* n_frames_out, void* stream);

/* ---- batched streaming flow: one session, several utterances ----------------------------------------------------------------
 * The reference serves concurrent streams one thread each, every chunk its own flow.inference call (cli/model.py:343-363).  A
 * multi-slot session holds n_slots utterances in one allocation (slot s, CFG branch c caches K/V rows from (2s + c) * cap), and
 * ONE chunk_batch call advances B distinct begun slots through one encoder / estimator pass, so B streams cost one chunk's
 * launches.  Slots in one call may sit at different chunk positions and have different prompt lengths and chunk lengths.
 * slots_create: kind 0 = CosyVoice2 U-Net (stage "flow"), 1 = CosyVoice3 DiT (stage "flow3"); max_frames per slot;
 * cvk_flow_stream_bytes reports the whole allocation.  cvk_flow_stream_create / cvk_flow3_stream_create are n_slots = 1,
 * cvk_flow_stream_begin is slot 0 and cvk_flow_stream_chunk a batch of one.
 * slot_begin: new utterance in `slot` (same arguments as cvk_flow_stream_begin).
 * chunk_batch: slots_host [B] distinct begun slots; tokens = the B token prefixes back to back (token_lens_host[b] each: prompt +
 * speech so far + 3 look-ahead, as for cvk_flow_stream_chunk); mel_out receives the new frames of every slot back to back
 * ([sum n_frames_out_host[b], 80], the ragged ABI convention), n_frames_out_host[b] their counts.  Every slot is checked (in
 * range, distinct, begun, both chunk ends on the 50-frame grid, capacity, mel_capacity_frames) before anything is launched: a
 * refused call returns CVK_ERR_INVALID and leaves every slot's state unchanged. */
int cvk_flow_stream_slots_create(cvk_ctx* ctx, int kind, int n_slots, int max_frames, int n_timesteps, cvk_flow_stream** out);
int cvk_flow_stream_slot_begin(cvk_ctx* ctx, cvk_flow_stream* fs, int slot, const float* prompt_feat, int prompt_frames,
                               const float* embedding, void* stream);
int cvk_flow_stream_chunk_batch(cvk_ctx* ctx, cvk_flow_stream* fs, int B, const int* slots_host, const int32_t* tokens,
                                const int* token_lens_host, float* mel_out, int mel_capacity_frames, int* n_frames_out_host,
                                void* stream);

/* ---- CosyVoice3 vocoder (stage "hift3") ------------------------------------------------------------------------------------
 * cosyvoice/hifigan/generator.py:572-726 CausalHiFTGenerator (+ f0_predictor.py:60-103 in float64, generator.py:716-717).
 * cvk_hift3_set_noise hands over the module's constructor-time random tensors, which are not state_dict entries
 * (generator.py:223-226): rand_ini [9] (SineGen2.rand_ini) and sine_noise [n][9] (SineGen2.sine_waves, indexed from the start of
 * every utterance).  cvk_hift3_inference = CausalHiFTGenerator.inference (:714-726) for B utterances: mel [sum T, 80] ->
 * wav [sum 480 T]; f0_out [sum T] and source_out [sum 480 T] are optional (NULL).  finalize == 0 is the streaming call
 * (:676-683, :709-710, :722-725): 3 + 4 mel frames of look-ahead are consumed and the last frame's samples dropped, i.e.
 * wav [sum 480 (T-8)], f0_out [sum (T-3)], source_out [sum 480 (T-3)]; every utterance needs T >= 9. */
int cvk_hift3_set_noise(cvk_ctx* ctx, const float* rand_ini, const float* sine_noise, long long n, int on_device);
int cvk_hift3_inference(cvk_ctx* ctx, const float* mel, const int* lens_host, int B, int finalize, float* wav, float* f0_out,
                        float* source_out, void* stream);

/* ---- CosyVoice3 flow (stage "flow3", cvk_finalize cfg = {DiT depth}) -----------------------------------------------------------
 * cosyvoice/flow/DiT/dit.py:145-176 (DiT.forward, the CFM estimator of CosyVoice3; TensorRT swap point flow_matching.py:126-153):
 * same dense argument layout as cvk_cfm_estimator - x, mu, cond [sum T, 80] time-major, t [B], spks [B, 80] -> out [sum T, 80];
 * streaming != 0 selects the static 50-frame block-causal mask (dit.py:165-166). */
int cvk_dit_estimator(cvk_ctx* ctx, const float* x, const float* mu, const float* t, const float* spks, const float* cond,
                      const int* lens_host, int B, int streaming, float* out, void* stream);
/* cosyvoice/flow/flow.py:369-414 CausalMaskedDiffWithDiT.inference for B utterances: tokens = prompt tokens followed by the new
 * tokens of every utterance (token_lens_host), prompt_feat [sum Tp, 80], embedding [B, 192]; finalize == 0: the last 3 tokens of
 * every utterance are look-ahead context (flow.py:389-392).  mel receives 2 * (tokens - context) - Tp frames per utterance.
 * The CFM noise is the tensor given to cvk_cfm_set_noise. */
int cvk_flow3_inference(cvk_ctx* ctx, const int32_t* tokens, const int* token_lens_host, const float* prompt_feat,
                        const int* prompt_feat_lens_host, const float* embedding, int B, int n_timesteps, int streaming, int finalize,
                        float* mel, void* stream);
/* the fixed noise tensor of CausalConditionalCFM (flow_matching.py:199-200) must be supplied once: [15000,80]
 * time-major (it is torch's seed-0 randn stream; the library does not re-implement torch's Philox/MT generator) */
int cvk_cfm_set_noise(cvk_ctx* ctx, const float* noise_tm, int T, int on_device);

/* ---------------------------------------------------------------------------------------------- speech-token LM
 * replaces cosyvoice/llm/llm.py:458-549 (Qwen2LM.inference / inference_wrapper; the vLLM swap point :506-534). */
typedef struct cvk_lm_session cvk_lm_session;
int cvk_lm_session_create(cvk_ctx* ctx, int max_batch, int max_context, cvk_lm_session** out);
void cvk_lm_session_destroy(cvk_ctx* ctx, cvk_lm_session* s);
/* llm.py:474-494: assemble [sos, embed(text), task_id, speech_embedding(prompt)] for B rows and run the prefill.
 * text [sum Nt] (prompt_text ++ text per row), speech [sum Np].  After the call the session holds the KV cache and
 * the hidden state of the last prompt position of every row. */
int cvk_lm_prefill(cvk_ctx* ctx, cvk_lm_session* s, const int32_t* text, const int* text_lens_host,
                   const int32_t* speech, const int* speech_lens_host, int B, void* stream);
/* llm.py:536-549: run up to n_steps decode steps for all live rows: head -> log_softmax -> RAS sampling ->
 * stop test -> next embedding.  uniforms [max_steps][B][2] (u1 nucleus draw, u2 fallback draw) indexed by the
 * absolute step; min_len/max_len [B] (device int32).  out_ids [B][out_ld] receives the accepted ids, out_count [B]
 * their number, done [B] (1 once a row hit a stop id or max_len).  Returns the number of live rows via
 * *live_host after synchronising the stream when live_host != NULL. */
int cvk_lm_decode(cvk_ctx* ctx, cvk_lm_session* s, int n_steps, const float* uniforms, const int32_t* min_len,
                  const int32_t* max_len, int32_t* out_ids, int out_ld, int32_t* out_count, int32_t* done, int* live_host,
                  void* stream);
/* teacher-forced log-probs for parity tests: embeds [sum L, 896] -> logp [sum L, V], V = cvk_lm_vocab */
int cvk_lm_forward_logp(cvk_ctx* ctx, const float* embeds, const int* lens_host, int B, float* logp, void* stream);
/* Width V of the log-prob / logits rows of the loaded LM: 6564 for Qwen2LM (llm.py:281), 6764 for CosyVoice3LM (llm.py:689: 6761
 * outputs, padded by 3 ids whose probability is exactly 0); 0 before the "llm" stage is finalised.  The "llm" stage recognises a
 * CosyVoice3LM state_dict by the absence of llm_embedding.weight. */
int cvk_lm_vocab(cvk_ctx* ctx);
/* Text-streaming LM (Qwen2LM.inference_bistream, llm.py:551-661: the caller interleaves 5 text : 15 speech embeddings and forces
 * fill tokens; cli/model.py:113-123 drives it when `text` is a generator).  cvk_lm_begin empties the session (B rows, normally 1);
 * cvk_lm_feed pushes n positions through the KV-cached decode path (llm.py:617-621 forward_one_step): ids_host / kinds_host are
 * HOST arrays, kind 0 = text id (embed_tokens), 1 = speech id (speech_embedding), 2 = llm_embedding row (0 sos, 1 task_id);
 * cvk_lm_next_logp writes log_softmax(llm_decoder(y_pred[:, -1])) (llm.py:622) of the last position to logp [B][V] (device, V = cvk_lm_vocab).
 * The draw itself is cvk_ras_sample (llm.py:627 sampling_ids). */
int cvk_lm_begin(cvk_ctx* ctx, cvk_lm_session* s, int B, void* stream);
int cvk_lm_feed(cvk_ctx* ctx, cvk_lm_session* s, const int32_t* ids_host, const int32_t* kinds_host, int n, void* stream);
int cvk_lm_next_logp(cvk_ctx* ctx, cvk_lm_session* s, float* logp, void* stream);
/* parity tests: the head logits [B][V] (llm_decoder output, llm.py:542, before log_softmax) that the most recent decode step
 * sampled from, copied to `logits` (device) */
int cvk_lm_last_logits(cvk_ctx* ctx, cvk_lm_session* s, float* logits, void* stream);
/* utils/common.py:138-167 + llm.py:150-160 as one kernel.  logp [B,V] (modified in place like the reference),
 * history [B, hist_ld] with hist_count [B] valid entries, uniforms [B,2], ignore_eos [B]; out ids [B]. */
int cvk_ras_sample(cvk_ctx* ctx, float* logp, int B, int V, const int32_t* history, int hist_ld, const int32_t* hist_count,
                   const float* uniforms, const int32_t* ignore_eos, int32_t* out_ids, void* stream);

/* ---------------------------------------------------------------------------------------------- mel frontend
 * replaces third_party/Matcha-TTS/matcha/utils/audio.py:45-82 with cosyvoice2.yaml:150-158 parameters (n_fft 1920, hop 480,
 * 80 mels, fmin 0, fmax 8000, center False).  wav [sum N_b] (24 kHz, any N_b >= 721: the reflect padding is taken about the true
 * last sample) -> mel [sum floor(N_b/480), 80] */
int cvk_mel_spectrogram(cvk_ctx* ctx, const float* wav, const int* lens_host, int B, float* mel, void* stream);
/* same with the filterbank's upper edge as a parameter: fmax_hz = 8000 (CosyVoice2) or 0 / 12000 = sr/2 (`fmax: null` of
 * examples/libritts/cosyvoice3/conf/cosyvoice3.yaml:140-147) */
int cvk_mel_spectrogram_ex(cvk_ctx* ctx, const float* wav, const int* lens_host, int B, int fmax_hz, float* mel, void* stream);

/* ---------------------------------------------------------------------------------------------- prompt-side features (16 kHz)
 * SURVEY 8(f) rank 2: the two feature extractors the reference frontend runs on the CPU before its ONNX sessions.
 * cvk_whisper_log_mel replaces whisper.log_mel_spectrogram(speech, n_mels=128) at cosyvoice/cli/frontend.py:98 (hann 400 / hop 160,
 * center, 128 Slaney mels, log10, floor at max - 8, (x + 4) / 4): wav [sum N_b] (N_b > 200) -> out [sum floor(N_b/160), 128],
 * time-major (the reference tensor [1,128,T] transposed).
 * cvk_kaldi_fbank replaces kaldi.fbank(speech, num_mel_bins=80, dither=0, sample_frequency=16000) at frontend.py:108-112 and, with
 * subtract_mean != 0, the mean normalisation of :113: wav [sum N_b] (N_b >= 400) -> out [sum 1 + floor((N_b-400)/160), 80].
 * The speech tokenizer / CAM++ networks that consume them are ONNX files outside the repository and are not rebuilt.
 * cvk_finalize(ctx, "prompt", NULL, 0) builds the constant DFT / filterbank matrices at set-up time (else: on the first call). */
int cvk_whisper_log_mel(cvk_ctx* ctx, const float* wav, const int* lens_host, int B, float* out, void* stream);
int cvk_kaldi_fbank(cvk_ctx* ctx, const float* wav, const int* lens_host, int B, int subtract_mean, float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CVK_H_ */
