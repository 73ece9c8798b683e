// extern "C" boundary of libcvk (include/cvk.h): argument checking, error translation, no exceptions across the ABI.
#include "common.cuh"
#include <string.h>

// stage entry points implemented in hift.cu / flow.cu / llm.cu / mel.cu
void hift_build(cvk_ctx* ctx);
void hift_f0(cvk_ctx* ctx, const float* mel, const int* lens, int B, float* f0_out, cudaStream_t st);
void hift_source(cvk_ctx* ctx, const float* f0, const int* lens, int B, const float* noise, float* source_out, cudaStream_t st);
void hift_decode(cvk_ctx* ctx, const float* mel, const int* lens, int B, const float* source, float* wav, cudaStream_t st);
void hift_inference(cvk_ctx* ctx, const float* mel, const int* lens, int B, const float* noise, const float* cache_source,
                    const int* cache_lens, float* wav, float* source_out, cudaStream_t st);
void flow_build(cvk_ctx* ctx, const int* cfg, int ncfg);
void flow_encoder(cvk_ctx* ctx, const int32_t* tokens, const int* lens, int B, int streaming, int context_len, float* h, cudaStream_t st);
void flow_estimator(cvk_ctx* ctx, const float* x, const float* mu, const float* t, const float* spks, const float* cond, const int* lens,
                    int B, int streaming, float* out, cudaStream_t st);
void flow_cfm_solve(cvk_ctx* ctx, const float* mu, const float* spks, const float* cond, const int* lens, int B, const float* z,
                    int n_timesteps, float cfg_rate, int streaming, float* out, cudaStream_t st);
void flow_inference(cvk_ctx* ctx, const int32_t* tokens, const int* token_lens, const float* prompt_feat, const int* prompt_feat_lens,
                    const float* embedding, int B, int n_timesteps, int streaming, int finalize, float* mel, cudaStream_t st);
void flow_set_noise(cvk_ctx* ctx, const float* noise_tm, int T, int on_device);
void llm_build(cvk_ctx* ctx, const int* cfg, int ncfg);
cvk_lm_session* llm_session_create(cvk_ctx* ctx, int max_batch, int max_context);
void llm_session_destroy(cvk_ctx* ctx, cvk_lm_session* s);
void hift3_build(cvk_ctx* ctx);
void hift3_set_noise(cvk_ctx* ctx, const float* rand_ini, const float* sine_noise, long long n, int on_device);
void hift3_inference(cvk_ctx* ctx, const float* mel, const int* lens, int B, int finalize, float* wav, float* f0_out, float* source_out,
                     cudaStream_t st);
void dit_build(cvk_ctx* ctx, const int* cfg, int ncfg);
void dit_estimator(cvk_ctx* ctx, const float* x, const float* mu, const float* t, const float* spks, const float* cond, const int* lens,
                   int B, int streaming, float* out, cudaStream_t st);
void flow3_inference(cvk_ctx* ctx, const int32_t* tokens, const int* token_lens, const float* prompt_feat, const int* prompt_feat_lens,
                     const float* embedding, int B, int n_timesteps, int streaming, int finalize, float* mel, cudaStream_t st);
void llm_prefill(cvk_ctx* ctx, cvk_lm_session* s, const int32_t* text, const int* text_lens, const int32_t* speech,
                 const int* speech_lens, int B, cudaStream_t st);
void llm_decode(cvk_ctx* ctx, cvk_lm_session* s, int n_steps, const float* uniforms, const int32_t* min_len, const int32_t* max_len,
                int32_t* out_ids, int out_ld, int32_t* out_count, int32_t* done, int* live_host, cudaStream_t st);
void llm_forward_logp(cvk_ctx* ctx, const float* embeds, const int* lens, int B, float* logp, cudaStream_t st);
void llm_last_logits(cvk_ctx* ctx, cvk_lm_session* s, float* logits, cudaStream_t st);
int llm_vocab(cvk_ctx* ctx);
void llm_session_begin(cvk_ctx* ctx, cvk_lm_session* s, int B, cudaStream_t st);
void llm_feed(cvk_ctx* ctx, cvk_lm_session* s, const int32_t* ids, const int32_t* kinds, int n, cudaStream_t st);
void llm_next_logp(cvk_ctx* ctx, cvk_lm_session* s, float* logp, cudaStream_t st);
void llm_ras_sample(cvk_ctx* ctx, float* logp, int B, int V, const int32_t* history, int hist_ld, const int32_t* hist_count,
                    const float* uniforms, const int32_t* ignore_eos, int32_t* out_ids, cudaStream_t st);
void mel_spectrogram(cvk_ctx* ctx, const float* wav, const int* lens, int B, int fmax_hz, float* mel, cudaStream_t st);
void mel_init(cvk_ctx* ctx);
void prompt_feat_init(cvk_ctx* ctx);

#define CVK_API_BEGIN            \
  if (!ctx) return CVK_ERR_INVALID; \
  try {                          \
    cudaSetDevice(ctx->device);
#define CVK_API_END                                  \
    return CVK_OK;                                   \
  } catch (const CvkError& e) {                      \
    ctx->last_error = e.what();                      \
    return e.code;                                   \
  } catch (const std::exception& e) {                \
    ctx->last_error = std::string("internal: ") + e.what(); \
    return CVK_ERR_INVALID;                          \
  }

extern "C" {

const char* cvk_version(void) { return "libcvk 0.1 (sm_100a)"; }

int cvk_create(int device, int precision, size_t workspace_bytes, cvk_ctx** out) {
  if (!out) return CVK_ERR_INVALID;
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= device || device < 0) return CVK_ERR_CUDA;   // no CPU fallback
  if (precision != CVK_PREC_FP32 && precision != CVK_PREC_BF16) return CVK_ERR_INVALID;
  if (cudaSetDevice(device) != cudaSuccess) return CVK_ERR_CUDA;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return CVK_ERR_CUDA;
  if (prop.major != 10) return CVK_ERR_CUDA;   // sm_100a only: the tcgen05/TMA kernels have no other code path
  cvk_ctx* ctx = new cvk_ctx();
  ctx->device = device;
  ctx->precision = precision;
  ctx->act_dtype = precision == CVK_PREC_BF16 ? DT_BF16 : DT_F32;
  ctx->num_sms = prop.multiProcessorCount;
  if (workspace_bytes == 0) workspace_bytes = (size_t)4 << 30;
  void* p = nullptr;
  if (cudaMalloc(&p, workspace_bytes) != cudaSuccess) {
    delete ctx;
    return CVK_ERR_OOM;
  }
  ctx->arena.base = (char*)p;
  ctx->arena.cap = workspace_bytes;
  *out = ctx;
  return CVK_OK;
}

void cvk_destroy(cvk_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  for (auto& kv : ctx->raw) cudaFree(kv.second.p);
  for (void* p : ctx->owned) cudaFree(p);
  cudaFree(ctx->arena.base);
  delete ctx;
}

const char* cvk_last_error(cvk_ctx* ctx) { return ctx ? ctx->last_error.c_str() : "null context"; }
thread_local int cvk_in_capture = 0;
int64_t cvk_launch_count(cvk_ctx* ctx) { return ctx ? ctx->launches.load() : 0; }
double cvk_last_op_ms(cvk_ctx* ctx) { return ctx ? ctx->op_ms : 0.0; }
int cvk_debug_read(cvk_ctx* ctx, long long* out, int n) {
  if (ctx && ctx->tl && out && n == 4096) {   // LM-chain timeline
    if (cudaMemcpy(out, ctx->tl, 4096 * sizeof(long long), cudaMemcpyDeviceToHost) != cudaSuccess) return CVK_ERR_CUDA;
    return CVK_OK;
  }
  if (!ctx || !ctx->dbg || !out || n > 1024) return CVK_ERR_INVALID;
  cudaSetDevice(ctx->device);
  if (cudaMemcpy(out, ctx->dbg, (size_t)n * sizeof(long long), cudaMemcpyDeviceToHost) != cudaSuccess) return CVK_ERR_CUDA;
  cudaMemset(ctx->dbg, 0, 1024 * sizeof(long long));
  return CVK_OK;
}

int cvk_set_option(cvk_ctx* ctx, const char* key, int value) {
  CVK_API_BEGIN
  std::string k(key ? key : "");
  if (k == "use_tc") ctx->use_tc = value;
  else if (k == "tc_bn256") ctx->tc_bn256 = value;
  else if (k == "tc_pbn256") ctx->tc_pbn256 = value;
  else if (k == "tc_epi") ctx->tc_epi = value;
  else if (k == "tc_persist") ctx->tc_persist = value;
  else if (k == "op_out_bf16") ctx->op_out_bf16 = value;
  else if (k == "op_iters") ctx->op_iters = value;
  else if (k == "use_graph") ctx->use_graph = value;
  else if (k == "use_tc_attn") ctx->use_tc_attn = value;
  else if (k == "use_skinny") ctx->use_skinny = value;
  else if (k == "lm_fused") ctx->lm_fused = value;
  else if (k == "pdl") ctx->pdl = value;
  else if (k == "lm_mega") ctx->lm_mega = value;
  else if (k == "attn_single_pass") ctx->attn_single_pass = value;
  else if (k == "enc_tc_attn") ctx->enc_tc_attn = value;
  else if (k == "hift_f16") ctx->hift_f16 = value;      // takes effect at the next cvk_finalize("hift" / "hift3")
  else if (k == "mega_coop") ctx->mega_coop = value;
  else if (k == "chain_timeline") {
    if (value && !ctx->tl) {
      ctx->tl = ctx->dmalloc(4096 * sizeof(long long));
      CVK_CHECK_CUDA(cudaMemset(ctx->tl, 0, 4096 * sizeof(long long)));
    }
    if (!value) ctx->tl = nullptr;
  }
  else if (k == "debug_timeline") {
    if (value && !ctx->dbg) {
      ctx->dbg = ctx->dmalloc(1024 * sizeof(long long));
      CVK_CHECK_CUDA(cudaMemset(ctx->dbg, 0, 1024 * sizeof(long long)));
    }
    if (!value) ctx->dbg = nullptr;
  }
  else throw CvkError(CVK_ERR_INVALID, "unknown option: " + k);
  CVK_API_END
}

int cvk_profile(cvk_ctx* ctx, int enable) {
  CVK_API_BEGIN
  CVK_CHECK_CUDA(cudaDeviceSynchronize());
  for (auto& r : ctx->prof) { ctx->event_pool.push_back(r.a); ctx->event_pool.push_back(r.b); }
  ctx->prof.clear();
  ctx->prof_on = enable;
  CVK_API_END
}

int cvk_profile_read(cvk_ctx* ctx, int family, double* ms, double* flops, double* bytes, int64_t* launches) {
  CVK_API_BEGIN
  CVK_REQUIRE(family >= 0 && family < FAM_COUNT && ms && flops && bytes && launches, "cvk_profile_read: bad arguments");
  CVK_CHECK_CUDA(cudaDeviceSynchronize());
  double t = 0, w = 0, by = 0;
  int64_t n = 0;
  for (auto& r : ctx->prof) {
    if (r.family != family) continue;
    float e = 0.f;
    CVK_CHECK_CUDA(cudaEventElapsedTime(&e, r.a, r.b));
    t += e; w += r.work; by += r.bytes; ++n;
  }
  *ms = t; *flops = w; *bytes = by; *launches = n;
  CVK_API_END
}

int cvk_set_tensor(cvk_ctx* ctx, const char* name, const float* data, int on_device, const int64_t* shape, int ndim) {
  CVK_API_BEGIN
  CVK_REQUIRE(name && data && shape && ndim >= 1 && ndim <= 4, "cvk_set_tensor: bad arguments");
  RawTensor t;
  t.shape.assign(shape, shape + ndim);
  size_t bytes = (size_t)t.numel() * sizeof(float);
  CVK_CHECK_CUDA(cudaMalloc((void**)&t.p, bytes));
  cudaError_t e = cudaMemcpy(t.p, data, bytes, on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    cudaFree(t.p);
    throw CvkError(CVK_ERR_CUDA, std::string("cvk_set_tensor copy: ") + cudaGetErrorString(e));
  }
  auto it = ctx->raw.find(name);
  if (it != ctx->raw.end()) {
    cudaFree(it->second.p);
    ctx->raw.erase(it);
  }
  ctx->raw[name] = t;
  CVK_API_END
}

int cvk_finalize(cvk_ctx* ctx, const char* stage, const int* cfg, int ncfg) {
  CVK_API_BEGIN
  std::string s(stage ? stage : "");
  if (s == "hift") hift_build(ctx);
  else if (s == "flow") flow_build(ctx, cfg, ncfg);
  else if (s == "flow3") dit_build(ctx, cfg, ncfg);
  else if (s == "hift3") hift3_build(ctx);
  else if (s == "llm") llm_build(ctx, cfg, ncfg);
  else if (s == "mel") mel_init(ctx);
  else if (s == "prompt") prompt_feat_init(ctx);
  else throw CvkError(CVK_ERR_INVALID, "unknown stage: " + s);
  CVK_CHECK_CUDA(cudaDeviceSynchronize());
  // raw tensors of this stage are no longer needed
  std::string prefix = s + ".";
  for (auto it = ctx->raw.begin(); it != ctx->raw.end();) {
    if (it->first.compare(0, prefix.size(), prefix) == 0) {
      cudaFree(it->second.p);
      it = ctx->raw.erase(it);
    } else ++it;
  }
  CVK_API_END
}

// ---------------------------------------------------------------------------------------------- generic ops
int cvk_op_conv1d(cvk_ctx* ctx, const float* x, const int* lens, int B, int K, const float* w, const float* bias, int N, int taps,
                  int dil, int shift0, int act, float* out, void* stream) {
  CVK_API_BEGIN
  cudaStream_t st = (cudaStream_t)stream;
  CVK_REQUIRE(x && lens && w && out && B > 0, "cvk_op_conv1d: bad arguments");
  ctx->arena.reset();
  size_t owned_mark = ctx->owned.size();
  int gap = 32;
  Seqs s = make_seqs(ctx, lens, B, gap, 1, 0, st);
  ConvW W = make_conv(ctx, w, bias, N, K, taps, dil, shift0);
  CVK_CHECK_CUDA(cudaDeviceSynchronize());   // weight repack runs on the default stream
  Mat a = arena_mat(ctx, ctx->act_dtype, s.R, K);
  zero_mat(ctx, st, a);
  pack_rows(ctx, st, x, K, s, a);
  Mat o = arena_mat(ctx, ctx->op_out_bf16 ? DT_BF16 : DT_F32, s.R, N);
  Epilogue e;
  e.act1 = act;
  e.act1_param = 0.1f;
  e.row2seq = s.d_row2seq;
  e.out = o;
  if (a.dtype == DT_BF16 && W.w16 == nullptr) {   // K not TMA-able: fp32 path
    Mat a32 = arena_mat(ctx, DT_F32, s.R, K);
    zero_mat(ctx, st, a32);
    pack_rows(ctx, st, x, K, s, a32);
    conv_gemm_simt(ctx, st, a32, W, e);
  } else {
    conv_gemm(ctx, st, a, W, e);
    if (ctx->op_iters > 0) {
      cudaEvent_t e0, e1;
      cudaEventCreate(&e0); cudaEventCreate(&e1);
      cudaEventRecord(e0, st);
      for (int i = 0; i < ctx->op_iters; ++i) conv_gemm(ctx, st, a, W, e);
      cudaEventRecord(e1, st);
      CVK_CHECK_CUDA(cudaStreamSynchronize(st));
      float ms = 0.f;
      cudaEventElapsedTime(&ms, e0, e1);
      ctx->op_ms = ms / ctx->op_iters;
      cudaEventDestroy(e0); cudaEventDestroy(e1);
    }
  }
  unpack_rows(ctx, st, o, s, 0, out, N);
  CVK_CHECK_CUDA(cudaStreamSynchronize(st));
  for (size_t i = owned_mark; i < ctx->owned.size(); ++i) cudaFree(ctx->owned[i]);
  ctx->owned.resize(owned_mark);
  CVK_API_END
}

// out[b, n] = sum_k x[b,k] w[n,k] (+bias) through the LM decode weight-streaming kernel (bf16 mode, rows <= 64)
int cvk_op_linear_small(cvk_ctx* ctx, const float* x, int rows, int K, const float* w, const float* bias, int N, float* out, int iters,
                        float* ms_out, long long* timeline_host, void* stream) {
  CVK_API_BEGIN
  cudaStream_t st = (cudaStream_t)stream;
  CVK_REQUIRE(x && w && out && rows > 0 && rows <= 64 && ctx->precision == CVK_PREC_BF16, "cvk_op_linear_small: bf16 context, rows <= 64");
  ctx->arena.reset();
  size_t owned_mark = ctx->owned.size();
  ConvW W = make_conv(ctx, w, bias, N, K, 1, 1, 0);
  skinny_tiled_weights(ctx, W);
  CVK_CHECK_CUDA(cudaDeviceSynchronize());
  Mat a32((void*)x, DT_F32, rows, K, K);
  Mat a = arena_mat(ctx, DT_BF16, rows, K);
  convert_mat(ctx, st, a32, a);
  Mat o(out, DT_F32, rows, N, N);
  size_t sf = skinny_scratch_floats(rows, N);
  float* scratch = (float*)ctx->arena.alloc(sf * sizeof(float));
  Epilogue e;
  e.out = o;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  conv_gemm_skinny(ctx, st, a, W, e, scratch, sf);
  cudaEventRecord(e0, st);
  for (int i = 0; i < iters; ++i) conv_gemm_skinny(ctx, st, a, W, e, scratch, sf);
  cudaEventRecord(e1, st);
  CVK_CHECK_CUDA(cudaStreamSynchronize(st));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, e0, e1);
  if (ms_out) *ms_out = iters > 0 ? ms / iters : 0.f;
  if (timeline_host && ctx->dbg) CVK_CHECK_CUDA(cudaMemcpy(timeline_host, ctx->dbg, 1024 * sizeof(long long), cudaMemcpyDeviceToHost));
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  ctx->tiled.erase(W.w16);
  for (size_t i = owned_mark; i < ctx->owned.size(); ++i) cudaFree(ctx->owned[i]);
  ctx->owned.resize(owned_mark);
  CVK_API_END
}

int cvk_op_attention(cvk_ctx* ctx, const float* q, const float* k, const float* v, const int* lens, int B, int H, int chunk,
                     float scale, float* out, void* stream) {
  CVK_API_BEGIN
  cudaStream_t st = (cudaStream_t)stream;
  CVK_REQUIRE(q && k && v && out && lens && B > 0 && H > 0, "cvk_op_attention: bad arguments");
  ctx->arena.reset();
  Seqs s = make_seqs(ctx, lens, B, 8, 1, 0, st);
  int C = H * 64;
  Mat mq = arena_mat(ctx, ctx->act_dtype, s.R, C), mk = arena_mat(ctx, ctx->act_dtype, s.R, C), mv = arena_mat(ctx, ctx->act_dtype, s.R, C);
  Mat mo = arena_mat(ctx, ctx->act_dtype, s.R, C);
  zero_mat(ctx, st, mq); zero_mat(ctx, st, mk); zero_mat(ctx, st, mv); zero_mat(ctx, st, mo);
  pack_rows(ctx, st, q, C, s, mq);
  pack_rows(ctx, st, k, C, s, mk);
  pack_rows(ctx, st, v, C, s, mv);
  attention_fwd(ctx, st, mq, mk, mv, s, H, chunk, scale, mo);
  unpack_rows(ctx, st, mo, s, 0, out, C);
  CVK_API_END
}

// ---------------------------------------------------------------------------------------------- HiFT
int cvk_hift_f0(cvk_ctx* ctx, const float* mel, const int* lens, int B, float* f0, void* stream) {
  CVK_API_BEGIN
  CVK_REQUIRE(mel && lens && f0 && B > 0, "cvk_hift_f0: bad arguments");
  hift_f0(ctx, mel, lens, B, f0, (cudaStream_t)stream);
  CVK_API_END
}
int cvk_hift_source(cvk_ctx* ctx, const float* f0, const int* lens, int B, const float* noise, float* source, void* stream) {
  CVK_API_BEGIN
  CVK_REQUIRE(f0 && lens && noise && source && B > 0, "cvk_hift_source: bad arguments");
  hift_source(ctx, f0, lens, B, noise, source, (cudaStream_t)stream);
  CVK_API_END
}
int cvk_hift_decode(cvk_ctx* ctx, const float* mel, const int* lens, int B, const float* source, float* wav, void* stream) {
  CVK_API_BEGIN
  CVK_REQUIRE(mel && lens && source && wav && B > 0, "cvk_hift_decode: bad arguments");
  hift_decode(ctx, mel, lens, B, source, wav, (cudaStream_t)stream);
  CVK_API_END
}
int cvk_hift_inference(cvk_ctx* ctx, const float* mel, const int* lens, int B, const float* noise, const float* cache_source,
                       const int* cache_lens, float* wav, float* source, void* stream) {
  CVK_API_BEGIN
  CVK_REQUIRE(mel && lens && noise && wav && B > 0, "cvk_hift_inference: bad arguments");
  hift_inference(ctx, mel, lens, B, noise, cache_source, cache_lens, wav, source, (cudaStream_t)stream);
  CVK_API_END
}

// ---------------------------------------------------------------------------------------------- flow
int cvk_flow_encoder(cvk_ctx* ctx, const int32_t* tokens, const int* lens, int B, int streaming, int context_len, float* h, void* stream) {
  CVK_API_BEGIN
  CVK_REQUIRE(tokens && lens && h && B > 0 && (context_len == 0 || context_len == 3), "cvk_flow_encoder: bad arguments");
  flow_encoder(ctx, tokens, lens, B, streaming, context_len, h, (cudaStream_t)stream);
  CVK_API_END
}
int cvk_cfm_estimator(cvk_ctx* ctx, const float* x, const float* mu, const float* t, const float* spks, const float* cond, const int* lens,
                      int B, int streaming, float* out, void* stream) {
  CVK_API_BEGIN
  CVK_REQUIRE(x && mu && t && spks && cond && lens && out && B > 0, "cvk_cfm_estimator: bad arguments");
  flow_estimator(ctx, x, mu, t, spks, cond, lens, B, streaming, out, (cudaStream_t)stream);
  CVK_API_END
}
int cvk_cfm_estimator_inplace(cvk_ctx* ctx, float* x, const float* mu, const float* t, const float* spks, const float* cond, const int* lens,
                              int B, int streaming, void* stream) {
  CVK_API_BEGIN
  CVK_REQUIRE(x && mu && t && spks && cond && lens && B > 0, "cvk_cfm_estimator_inplace: bad arguments");
  flow_estimator(ctx, x, mu, t, spks, cond, lens, B, streaming, x, (cudaStream_t)stream);     // x is packed before the first write
  CVK_API_END
}
int cvk_workspace_bytes(cvk_ctx* ctx, size_t* capacity, size_t* high_water) {
  CVK_API_BEGIN
  CVK_REQUIRE(capacity && high_water, "cvk_workspace_bytes: bad arguments");
  *capacity = ctx->arena.cap;
  *high_water = ctx->arena.high;
  CVK_API_END
}
int cvk_cfm_solve(cvk_ctx* ctx, const float* mu, const float* spks, const float* cond, const int* lens, int B, const float* z,
                  int n_timesteps, float cfg_rate, int streaming, float* out, void* stream) {
  CVK_API_BEGIN
  CVK_REQUIRE(mu && spks && cond && lens && out && B > 0 && n_timesteps > 0, "cvk_cfm_solve: bad arguments");
  flow_cfm_solve(ctx, mu, spks, cond, lens, B, z, n_timesteps, cfg_rate, streaming, out, (cudaStream_t)stream);
  CVK_API_END
}
int cvk_flow_inference(cvk_ctx* ctx, const int32_t* tokens, const int* token_lens, const float* prompt_feat, const int* prompt_feat_lens,
                       const float* embedding, int B, int n_timesteps, int streaming, int finalize, float* mel, void* stream) {
  CVK_API_BEGIN
  CVK_REQUIRE(tokens && token_lens && prompt_feat_lens && embedding && mel && B > 0, "cvk_flow_inference: bad arguments");
  flow_inference(ctx, tokens, token_lens, prompt_feat, prompt_feat_lens, embedding, B, n_timesteps, streaming, finalize, mel,
                 (cudaStream_t)stream);
  CVK_API_END
}
int cvk_flow_stream_slots_create(cvk_ctx* ctx, int kind, int n_slots, int max_frames, int n_timesteps, cvk_flow_stream** out) {
  CVK_API_BEGIN
  CVK_REQUIRE(out != nullptr, "cvk_flow_stream_slots_create: bad arguments");
  *out = flow_stream_create(ctx, kind, n_slots, max_frames, n_timesteps);
  CVK_API_END
}
int cvk_flow_stream_create(cvk_ctx* ctx, int max_frames, int n_timesteps, cvk_flow_stream** out) {
  return cvk_flow_stream_slots_create(ctx, 0, 1, max_frames, n_timesteps, out);
}
int cvk_flow3_stream_create(cvk_ctx* ctx, int max_frames, int n_timesteps, cvk_flow_stream** out) {
  return cvk_flow_stream_slots_create(ctx, 1, 1, max_frames, n_timesteps, out);
}
void cvk_flow_stream_destroy(cvk_ctx* ctx, cvk_flow_stream* fs) {
  if (!ctx || !fs) return;
  try { cudaSetDevice(ctx->device); flow_stream_destroy(fs); } catch (...) {}
}
long long cvk_flow_stream_bytes(const cvk_flow_stream* fs) { return fs ? (long long)flow_stream_bytes(fs) : 0; }
int cvk_flow_stream_slot_begin(cvk_ctx* ctx, cvk_flow_stream* fs, int slot, const float* prompt_feat, int prompt_frames, const float* embedding,
                               void* stream) {
  CVK_API_BEGIN
  CVK_REQUIRE(fs && embedding && (prompt_feat || prompt_frames == 0), "cvk_flow_stream_slot_begin: bad arguments");
  flow_stream_begin(ctx, fs, slot, prompt_feat, prompt_frames, embedding, (cudaStream_t)stream);
  CVK_API_END
}
int cvk_flow_stream_begin(cvk_ctx* ctx, cvk_flow_stream* fs, const float* prompt_feat, int prompt_frames, const float* embedding, void* stream) {
  return cvk_flow_stream_slot_begin(ctx, fs, 0, prompt_feat, prompt_frames, embedding, stream);
}
int cvk_flow_stream_chunk_batch(cvk_ctx* ctx, cvk_flow_stream* fs, int B, const int* slots_host, const int32_t* tokens,
                                const int* token_lens_host, float* mel_out, int mel_capacity_frames, int* n_frames_out_host, void* stream) {
  CVK_API_BEGIN
  CVK_REQUIRE(fs && B > 0 && slots_host && tokens && token_lens_host && mel_out && n_frames_out_host, "cvk_flow_stream_chunk_batch: bad arguments");
  for (int b = 0; b < B; ++b) CVK_REQUIRE(token_lens_host[b] > 3, "cvk_flow_stream_chunk_batch: a prefix without its 3 look-ahead tokens");
  flow_stream_chunk_batch(ctx, fs, B, slots_host, tokens, token_lens_host, mel_out, mel_capacity_frames, n_frames_out_host, (cudaStream_t)stream);
  CVK_API_END
}
int cvk_flow_stream_chunk(cvk_ctx* ctx, cvk_flow_stream* fs, const int32_t* tokens, int n_tokens, float* mel_out, int mel_capacity_frames,
                          int* n_frames_out, void* stream) {
  const int slot = 0;
  return cvk_flow_stream_chunk_batch(ctx, fs, 1, &slot, tokens, &n_tokens, mel_out, mel_capacity_frames, n_frames_out, stream);
}
int cvk_cfm_set_noise(cvk_ctx* ctx, const float* noise_tm, int T, int on_device) {
  CVK_API_BEGIN
  CVK_REQUIRE(noise_tm && T > 0, "cvk_cfm_set_noise: bad arguments");
  flow_set_noise(ctx, noise_tm, T, on_device);
  CVK_API_END
}

// ---------------------------------------------------------------------------------------------- LM
int cvk_hift3_set_noise(cvk_ctx* ctx, const float* rand_ini, const float* sine_noise, long long n, int on_device) {
  CVK_API_BEGIN
  CVK_REQUIRE(rand_ini && sine_noise && n > 0, "cvk_hift3_set_noise: bad arguments");
  hift3_set_noise(ctx, rand_ini, sine_noise, n, on_device);
  CVK_API_END
}
int cvk_hift3_inference(cvk_ctx* ctx, const float* mel, const int* lens_host, int B, int finalize, float* wav, float* f0_out,
                        float* source_out, void* stream) {
  CVK_API_BEGIN
  CVK_REQUIRE(mel && lens_host && wav && B > 0, "cvk_hift3_inference: bad arguments");
  hift3_inference(ctx, mel, lens_host, B, finalize, wav, f0_out, source_out, (cudaStream_t)stream);
  CVK_API_END
}
int cvk_dit_estimator(cvk_ctx* ctx, const float* x, const float* mu, const float* t, const float* spks, const float* cond,
                      const int* lens_host, int B, int streaming, float* out, void* stream) {
  CVK_API_BEGIN
  CVK_REQUIRE(x && mu && t && spks && cond && lens_host && out && B > 0, "cvk_dit_estimator: bad arguments");
  dit_estimator(ctx, x, mu, t, spks, cond, lens_host, B, streaming, out, (cudaStream_t)stream);
  CVK_API_END
}
int cvk_flow3_inference(cvk_ctx* ctx, const int32_t* tokens, const int* token_lens_host, const float* prompt_feat,
                        const int* prompt_feat_lens_host, const float* embedding, int B, int n_timesteps, int streaming, int finalize,
                        float* mel, void* stream) {
  CVK_API_BEGIN
  CVK_REQUIRE(tokens && token_lens_host && prompt_feat_lens_host && embedding && mel && B > 0 && n_timesteps > 0,
              "cvk_flow3_inference: bad arguments");
  flow3_inference(ctx, tokens, token_lens_host, prompt_feat, prompt_feat_lens_host, embedding, B, n_timesteps, streaming, finalize, mel,
                  (cudaStream_t)stream);
  CVK_API_END
}
int cvk_lm_session_create(cvk_ctx* ctx, int max_batch, int max_context, cvk_lm_session** out) {
  CVK_API_BEGIN
  CVK_REQUIRE(out && max_batch > 0 && max_context > 0, "cvk_lm_session_create: bad arguments");
  *out = llm_session_create(ctx, max_batch, max_context);
  CVK_API_END
}
void cvk_lm_session_destroy(cvk_ctx* ctx, cvk_lm_session* s) {
  if (!ctx || !s) return;
  try { llm_session_destroy(ctx, s); } catch (...) {}
}
int cvk_lm_prefill(cvk_ctx* ctx, cvk_lm_session* s, const int32_t* text, const int* text_lens, const int32_t* speech,
                   const int* speech_lens, int B, void* stream) {
  CVK_API_BEGIN
  CVK_REQUIRE(s && text && text_lens && speech_lens && B > 0, "cvk_lm_prefill: bad arguments");
  llm_prefill(ctx, s, text, text_lens, speech, speech_lens, B, (cudaStream_t)stream);
  CVK_API_END
}
int cvk_lm_decode(cvk_ctx* ctx, cvk_lm_session* s, int n_steps, const float* uniforms, const int32_t* min_len, const int32_t* max_len,
                  int32_t* out_ids, int out_ld, int32_t* out_count, int32_t* done, int* live_host, void* stream) {
  CVK_API_BEGIN
  CVK_REQUIRE(s && uniforms && min_len && max_len && out_ids && out_count && done && n_steps >= 0, "cvk_lm_decode: bad arguments");
  llm_decode(ctx, s, n_steps, uniforms, min_len, max_len, out_ids, out_ld, out_count, done, live_host, (cudaStream_t)stream);
  CVK_API_END
}
int cvk_lm_forward_logp(cvk_ctx* ctx, const float* embeds, const int* lens, int B, float* logp, void* stream) {
  CVK_API_BEGIN
  CVK_REQUIRE(embeds && lens && logp && B > 0, "cvk_lm_forward_logp: bad arguments");
  llm_forward_logp(ctx, embeds, lens, B, logp, (cudaStream_t)stream);
  CVK_API_END
}
int cvk_lm_vocab(cvk_ctx* ctx) { return ctx ? llm_vocab(ctx) : 0; }
int cvk_lm_begin(cvk_ctx* ctx, cvk_lm_session* s, int B, void* stream) {
  CVK_API_BEGIN
  CVK_REQUIRE(s != nullptr, "cvk_lm_begin: bad arguments");
  llm_session_begin(ctx, s, B, (cudaStream_t)stream);
  CVK_API_END
}
int cvk_lm_feed(cvk_ctx* ctx, cvk_lm_session* s, const int32_t* ids_host, const int32_t* kinds_host, int n, void* stream) {
  CVK_API_BEGIN
  CVK_REQUIRE(s && ids_host && kinds_host && n > 0, "cvk_lm_feed: bad arguments");
  llm_feed(ctx, s, ids_host, kinds_host, n, (cudaStream_t)stream);
  CVK_API_END
}
int cvk_lm_next_logp(cvk_ctx* ctx, cvk_lm_session* s, float* logp, void* stream) {
  CVK_API_BEGIN
  CVK_REQUIRE(s && logp, "cvk_lm_next_logp: bad arguments");
  llm_next_logp(ctx, s, logp, (cudaStream_t)stream);
  CVK_API_END
}
int cvk_lm_last_logits(cvk_ctx* ctx, cvk_lm_session* s, float* logits, void* stream) {
  CVK_API_BEGIN
  CVK_REQUIRE(s && logits, "cvk_lm_last_logits: bad arguments");
  llm_last_logits(ctx, s, logits, (cudaStream_t)stream);
  CVK_API_END
}
int cvk_ras_sample(cvk_ctx* ctx, float* logp, int B, int V, const int32_t* history, int hist_ld, const int32_t* hist_count,
                   const float* uniforms, const int32_t* ignore_eos, int32_t* out_ids, void* stream) {
  CVK_API_BEGIN
  CVK_REQUIRE(logp && history && hist_count && uniforms && ignore_eos && out_ids && B > 0 && V > 0, "cvk_ras_sample: bad arguments");
  llm_ras_sample(ctx, logp, B, V, history, hist_ld, hist_count, uniforms, ignore_eos, out_ids, (cudaStream_t)stream);
  CVK_API_END
}

// ---------------------------------------------------------------------------------------------- mel
int cvk_mel_spectrogram(cvk_ctx* ctx, const float* wav, const int* lens, int B, float* mel, void* stream) {
  CVK_API_BEGIN
  CVK_REQUIRE(wav && lens && mel && B > 0, "cvk_mel_spectrogram: bad arguments");
  mel_spectrogram(ctx, wav, lens, B, 8000, mel, (cudaStream_t)stream);
  CVK_API_END
}
int cvk_mel_spectrogram_ex(cvk_ctx* ctx, const float* wav, const int* lens, int B, int fmax_hz, float* mel, void* stream) {
  CVK_API_BEGIN
  CVK_REQUIRE(wav && lens && mel && B > 0, "cvk_mel_spectrogram_ex: bad arguments");
  mel_spectrogram(ctx, wav, lens, B, fmax_hz, mel, (cudaStream_t)stream);
  CVK_API_END
}
int cvk_whisper_log_mel(cvk_ctx* ctx, const float* wav, const int* lens, int B, float* out, void* stream) {
  CVK_API_BEGIN
  CVK_REQUIRE(wav && lens && out && B > 0, "cvk_whisper_log_mel: bad arguments");
  whisper_log_mel(ctx, wav, lens, B, out, (cudaStream_t)stream);
  CVK_API_END
}
int cvk_kaldi_fbank(cvk_ctx* ctx, const float* wav, const int* lens, int B, int subtract_mean, float* out, void* stream) {
  CVK_API_BEGIN
  CVK_REQUIRE(wav && lens && out && B > 0, "cvk_kaldi_fbank: bad arguments");
  kaldi_fbank80(ctx, wav, lens, B, subtract_mean, out, (cudaStream_t)stream);
  CVK_API_END
}

}  // extern "C"
