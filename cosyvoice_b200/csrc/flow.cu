// CosyVoice2 flow stage: speech tokens -> mel (conformer up-sampling encoder + conditional flow matching with a
// causal U-Net estimator), batched over ragged utterances.
//
// Follows cosyvoice/flow/flow.py:235-281 (CausalMaskedDiffWithXvec.inference),
// cosyvoice/transformer/upsample_encoder.py:244-307 (+ subsampling.py:92-113, embedding.py:224-302,
// encoder_layer.py:160-236, attention.py:249-330), cosyvoice/flow/flow_matching.py:203-227 + 71-124 (Euler + CFG),
// cosyvoice/flow/decoder.py:405-494 with Matcha decoder.py:14-117 / transformer.py:243-316;
// hyper-parameters examples/libritts/cosyvoice2/conf/cosyvoice2.yaml:38-87.
//
// Design: everything is a time-major [rows, channels] matrix, so the reference's b c t <-> b t c rearranges vanish;
// channel concatenations (pack([x, mu, spks, cond]) and the U-Net skip) are column slices of one wide buffer;
// masks are row predicates; the two CFG branches are simply 2B sequences of one ragged batch.
#include "common.cuh"
#include <math.h>

namespace {
constexpr int D_ENC = 512, H_ENC = 8, FF_ENC = 2048;
constexpr int C_EST = 256, H_EST = 8, N_MEL = 80, TEMB = 1024;
constexpr int CHUNK_TOK = 25;   // cosyvoice2.yaml:16 static chunk (tokens); 50 after the x2 up-sampler and for mel frames

struct EncLayerW {
  float *ln1_g, *ln1_b, *ln2_g, *ln2_b;
  ConvW qkv, out, pos, w1, w2;
  float *bias_u, *bias_v;
};
struct EmbedW {
  ConvW lin;
  float *ln_g, *ln_b;
};
struct ResnetW {
  ConvW c1, c2, res;
  float *ln1_g, *ln1_b, *ln2_g, *ln2_b;
};
struct TBlockW {
  float *ln1_g, *ln1_b, *ln3_g, *ln3_b;
  ConvW qkv, out, ff1, ff2;
};
struct StageW {
  ResnetW rn;
  std::vector<TBlockW> tb;
};
}  // namespace

struct FlowModel {
  int enc_blocks = 6, enc_up_blocks = 4, num_mid = 12, n_blocks = 4;
  float* tok_emb = nullptr;       // [6561][512]
  ConvW spk_affine;               // 192 -> 80
  EmbedW embed, up_embed;
  ConvW pre1, pre2, up_conv, enc_proj;
  float *after_g, *after_b;
  std::vector<EncLayerW> enc, enc_up;
  // estimator
  ConvW t1, t2, tmlp_all;         // time MLP; all 14 resnet time projections concatenated [14*256][1024]
  std::vector<StageW> stages;     // down, mid x num_mid, up
  ConvW down_conv, up_conv2, final_conv, final_proj;
  float *final_g, *final_b;
  float* noise = nullptr;         // [T][80] time-major copy of CausalConditionalCFM.rand_noise
  int noise_T = 0;
};

// Streaming synthesis sessions of the flow stage (cvk_flow_stream_*): the caches that let a chunk call compute ONLY its new
// frames, for n_slots utterances in one allocation.  Per Euler step: K/V rows of every estimator transformer block for both CFG
// sequences of every slot (slot s, branch c at rows (2s + c) * cap), and the tails of every causal convolution's input.
struct cvk_flow_stream {
  int kind = 0;                 // 0: CosyVoice2 U-Net estimator (stage "flow"), 1: CosyVoice3 DiT (stage "flow3")
  int kv_width = 1024;          // K | V columns per cached row: 2 x 512 (U-Net blocks), 2 x 1024 (DiT blocks)
  int tail_rows = 2;            // rows a causal convolution reads in front of a chunk: k3 -> 2, the DiT's k31 position convolutions -> 30
  int conv_c = 512;             // widest convolution input
  int cap = 0, n_slots = 1, n_steps = 0, adt = DT_F32, n_tb = 0, n_conv = 0;
  void* kv = nullptr;           // per step: [n_tb][n_slots * 2 * cap + 64][kv_width]
  void* conv = nullptr;         // per step: [n_conv][n_slots * 2][tail_rows][conv_c]
  size_t kv_step_bytes = 0, conv_step_bytes = 0;
  std::vector<int> frames_done; // per slot: mel frames (prompt included) already produced
  std::vector<int> prompt_frames;
  std::vector<char> begun;
  float* prompt_feat = nullptr; // [n_slots][cap][80]
  float* spk = nullptr;         // [n_slots][80] projected speaker embeddings
  int* d_geo = nullptr;         // per sequence of a call (2 per slot): kstart | klen | qoff | conv state index, 2 * n_slots each
  KvGeom kg;
  const int* d_cidx = nullptr;
};

namespace {

float* copy_param(cvk_ctx* ctx, const std::string& name) {
  const RawTensor& t = ctx->get_raw(name);
  return dev_copy_f32(ctx, t.p, (size_t)t.numel());
}

// concatenate Linear weights (rows) [N_i][K] -> [sum N_i][K]
ConvW concat_linear(cvk_ctx* ctx, const std::vector<std::string>& wnames, const std::vector<std::string>& bnames) {
  int K = (int)ctx->get_raw(wnames[0]).shape[1];
  int N = 0;
  for (auto& n : wnames) N += (int)ctx->get_raw(n).shape[0];
  ConvW w;
  w.N = N; w.K = K; w.taps = 1; w.dil = 1; w.shift0 = 0;
  w.w32 = (float*)ctx->dmalloc((size_t)N * K * sizeof(float));
  size_t off = 0;
  for (auto& n : wnames) {
    const RawTensor& t = ctx->get_raw(n);
    CVK_CHECK_CUDA(cudaMemcpy(w.w32 + off, t.p, (size_t)t.numel() * sizeof(float), cudaMemcpyDeviceToDevice));
    off += t.numel();
  }
  if (!bnames.empty()) {
    w.bias = (float*)ctx->dmalloc((size_t)N * sizeof(float));
    size_t bo = 0;
    for (auto& n : bnames) {
      const RawTensor& t = ctx->get_raw(n);
      CVK_CHECK_CUDA(cudaMemcpy(w.bias + bo, t.p, (size_t)t.numel() * sizeof(float), cudaMemcpyDeviceToDevice));
      bo += t.numel();
    }
  }
  finish_convw(ctx, w);
  return w;
}

// nearest x2 up-sampling + left pad 4 + Conv1d(k5) (upsample_encoder.py:59-63) as a 3-tap polyphase conv on the
// un-upsampled input: out[2t+ph] = sum_m x[t-2+m] * Wp[ph][m],  Wp[0] = {w0+w1, w2+w3, w4}, Wp[1] = {w0, w1+w2, w3+w4}
__global__ void upsample_poly_kernel(const float* __restrict__ w /*[N][K][5]*/, float* __restrict__ o /*[2N][3][K]*/, int N, int K) {
  size_t total = (size_t)2 * N * 3 * K;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    int k = i % K;
    int m = (i / K) % 3;
    int n2 = i / ((size_t)K * 3);
    int ph = n2 / N, n = n2 % N;
    const float* wp = w + ((size_t)n * K + k) * 5;
    float v;
    if (ph == 0) v = m == 0 ? wp[0] + wp[1] : (m == 1 ? wp[2] + wp[3] : wp[4]);
    else v = m == 0 ? wp[0] : (m == 1 ? wp[1] + wp[2] : wp[3] + wp[4]);
    o[i] = v;
  }
}
__global__ void repeat2_kernel(const float* __restrict__ b, float* __restrict__ o, int N) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < 2 * N) o[i] = b[i % N];
}

EncLayerW build_enc_layer(cvk_ctx* ctx, const std::string& p) {
  EncLayerW l;
  l.ln1_g = copy_param(ctx, p + ".norm_mha.weight");
  l.ln1_b = copy_param(ctx, p + ".norm_mha.bias");
  l.ln2_g = copy_param(ctx, p + ".norm_ff.weight");
  l.ln2_b = copy_param(ctx, p + ".norm_ff.bias");
  std::string a = p + ".self_attn";
  l.qkv = concat_linear(ctx, {a + ".linear_q.weight", a + ".linear_k.weight", a + ".linear_v.weight"},
                        {a + ".linear_q.bias", a + ".linear_k.bias", a + ".linear_v.bias"});
  l.out = make_linear(ctx, a + ".linear_out.weight", a + ".linear_out.bias");
  l.pos = make_linear(ctx, a + ".linear_pos.weight", "");
  l.bias_u = copy_param(ctx, a + ".pos_bias_u");
  l.bias_v = copy_param(ctx, a + ".pos_bias_v");
  l.w1 = make_linear(ctx, p + ".feed_forward.w_1.weight", p + ".feed_forward.w_1.bias");
  l.w2 = make_linear(ctx, p + ".feed_forward.w_2.weight", p + ".feed_forward.w_2.bias");
  return l;
}

EmbedW build_embed(cvk_ctx* ctx, const std::string& p) {
  EmbedW e;
  e.lin = make_linear(ctx, p + ".out.0.weight", p + ".out.0.bias");
  e.ln_g = copy_param(ctx, p + ".out.1.weight");
  e.ln_b = copy_param(ctx, p + ".out.1.bias");
  return e;
}

ResnetW build_resnet(cvk_ctx* ctx, const std::string& p) {
  ResnetW r;
  r.c1 = make_conv_named(ctx, p + ".block1.block.0.weight", p + ".block1.block.0.bias", 1, -2);
  r.c2 = make_conv_named(ctx, p + ".block2.block.0.weight", p + ".block2.block.0.bias", 1, -2);
  r.res = make_conv_named(ctx, p + ".res_conv.weight", p + ".res_conv.bias", 1, 0);
  r.ln1_g = copy_param(ctx, p + ".block1.block.2.weight");
  r.ln1_b = copy_param(ctx, p + ".block1.block.2.bias");
  r.ln2_g = copy_param(ctx, p + ".block2.block.2.weight");
  r.ln2_b = copy_param(ctx, p + ".block2.block.2.bias");
  return r;
}

TBlockW build_tblock(cvk_ctx* ctx, const std::string& p) {
  TBlockW t;
  t.ln1_g = copy_param(ctx, p + ".norm1.weight");
  t.ln1_b = copy_param(ctx, p + ".norm1.bias");
  t.ln3_g = copy_param(ctx, p + ".norm3.weight");
  t.ln3_b = copy_param(ctx, p + ".norm3.bias");
  t.qkv = concat_linear(ctx, {p + ".attn1.to_q.weight", p + ".attn1.to_k.weight", p + ".attn1.to_v.weight"}, {});
  t.out = make_linear(ctx, p + ".attn1.to_out.0.weight", p + ".attn1.to_out.0.bias");
  t.ff1 = make_linear(ctx, p + ".ff.net.0.proj.weight", p + ".ff.net.0.proj.bias");
  t.ff2 = make_linear(ctx, p + ".ff.net.2.weight", p + ".ff.net.2.bias");
  return t;
}

StageW build_stage(cvk_ctx* ctx, const std::string& p, int n_blocks) {
  StageW s;
  s.rn = build_resnet(ctx, p + ".0");
  for (int j = 0; j < n_blocks; ++j) s.tb.push_back(build_tblock(ctx, p + ".1." + std::to_string(j)));
  return s;
}

}  // namespace

void flow_build(cvk_ctx* ctx, const int* cfg, int ncfg) {
  FlowModel* m = new FlowModel();
  if (ncfg >= 4) {
    m->enc_blocks = cfg[0]; m->enc_up_blocks = cfg[1]; m->num_mid = cfg[2]; m->n_blocks = cfg[3];
  }
  const std::string P = "flow.";
  m->tok_emb = copy_param(ctx, P + "input_embedding.weight");
  m->spk_affine = make_linear(ctx, P + "spk_embed_affine_layer.weight", P + "spk_embed_affine_layer.bias");
  m->spk_affine.w16 = nullptr;   // tiny, fp32
  const std::string E = P + "encoder.";
  m->embed = build_embed(ctx, E + "embed");
  m->up_embed = build_embed(ctx, E + "up_embed");
  m->pre1 = make_conv_named(ctx, E + "pre_lookahead_layer.conv1.weight", E + "pre_lookahead_layer.conv1.bias", 1, 0);
  m->pre2 = make_conv_named(ctx, E + "pre_lookahead_layer.conv2.weight", E + "pre_lookahead_layer.conv2.bias", 1, -2);
  {
    const RawTensor& w = ctx->get_raw(E + "up_layer.conv.weight");
    int N = (int)w.shape[0], K = (int)w.shape[1];
    CVK_REQUIRE(w.shape[2] == 5, "up_layer.conv must have kernel 5");
    ConvW c;
    c.N = 2 * N; c.K = K; c.taps = 3; c.dil = 1; c.shift0 = -2;
    c.w32 = (float*)ctx->dmalloc((size_t)c.N * 3 * K * sizeof(float));
    upsample_poly_kernel<<<256, 256>>>(w.p, c.w32, N, K);
    CVK_LAUNCH_CHECK();
    c.bias = (float*)ctx->dmalloc((size_t)c.N * sizeof(float));
    repeat2_kernel<<<ceil_div(2 * N, 256), 256>>>(ctx->get_raw(E + "up_layer.conv.bias").p, c.bias, N);
    CVK_LAUNCH_CHECK();
    finish_convw(ctx, c);
    m->up_conv = c;
  }
  m->after_g = copy_param(ctx, E + "after_norm.weight");
  m->after_b = copy_param(ctx, E + "after_norm.bias");
  for (int i = 0; i < m->enc_blocks; ++i) m->enc.push_back(build_enc_layer(ctx, E + "encoders." + std::to_string(i)));
  for (int i = 0; i < m->enc_up_blocks; ++i) m->enc_up.push_back(build_enc_layer(ctx, E + "up_encoders." + std::to_string(i)));
  m->enc_proj = make_linear(ctx, P + "encoder_proj.weight", P + "encoder_proj.bias");
  const std::string D = P + "decoder.estimator.";
  m->t1 = make_linear(ctx, D + "time_mlp.linear_1.weight", D + "time_mlp.linear_1.bias");
  m->t2 = make_linear(ctx, D + "time_mlp.linear_2.weight", D + "time_mlp.linear_2.bias");
  m->t1.w16 = nullptr;
  m->t2.w16 = nullptr;
  std::vector<std::string> stage_names;
  stage_names.push_back(D + "down_blocks.0");
  for (int i = 0; i < m->num_mid; ++i) stage_names.push_back(D + "mid_blocks." + std::to_string(i));
  stage_names.push_back(D + "up_blocks.0");
  {
    std::vector<std::string> wn, bn;
    for (auto& s : stage_names) {
      wn.push_back(s + ".0.mlp.1.weight");
      bn.push_back(s + ".0.mlp.1.bias");
    }
    m->tmlp_all = concat_linear(ctx, wn, bn);
    m->tmlp_all.w16 = nullptr;
  }
  for (auto& s : stage_names) m->stages.push_back(build_stage(ctx, s, m->n_blocks));
  m->down_conv = make_conv_named(ctx, D + "down_blocks.0.2.weight", D + "down_blocks.0.2.bias", 1, -2);
  m->up_conv2 = make_conv_named(ctx, D + "up_blocks.0.2.weight", D + "up_blocks.0.2.bias", 1, -2);
  m->final_conv = make_conv_named(ctx, D + "final_block.block.0.weight", D + "final_block.block.0.bias", 1, -2);
  m->final_g = copy_param(ctx, D + "final_block.block.2.weight");
  m->final_b = copy_param(ctx, D + "final_block.block.2.bias");
  m->final_proj = make_conv_named(ctx, D + "final_proj.weight", D + "final_proj.bias", 1, 0);
  CVK_CHECK_CUDA(cudaDeviceSynchronize());
  if (ctx->flow && ctx->flow->noise) {   // keep a previously supplied noise tensor
    m->noise = ctx->flow->noise;
    m->noise_T = ctx->flow->noise_T;
  }
  ctx->flow = m;
}

void flow_set_noise(cvk_ctx* ctx, const float* noise_tm, int T, int on_device) {
  if (!ctx->flow) ctx->flow = new FlowModel();
  FlowModel* m = ctx->flow;
  m->noise = (float*)ctx->dmalloc((size_t)T * N_MEL * sizeof(float));
  CVK_CHECK_CUDA(cudaMemcpy(m->noise, noise_tm, (size_t)T * N_MEL * sizeof(float), on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice));
  m->noise_T = T;
}

// ================================================================================================ kernels
namespace {

// token ids -> embedding rows (flow.py:252-254: clamp(min=0), padding mask), written as the Linear operand
template <typename TO>
__global__ void token_embed_kernel(const int32_t* __restrict__ tokens, const int* __restrict__ tok_off, const float* __restrict__ table,
                                   const int* __restrict__ start, const int* __restrict__ len, TO* __restrict__ out, int ldo,
                                   int width = D_ENC) {
  int b = blockIdx.y;
  int L = len[b];
  for (int t = blockIdx.x; t < L; t += gridDim.x) {
    int id = tokens[tok_off[b] + t];
    if (id < 0) id = 0;
    const float* src = table + (size_t)id * width;
    TO* dst = out + (size_t)(start[b] + t) * ldo;
    for (int c = threadIdx.x; c < width; c += blockDim.x) dst[c] = from_f32<TO>(src[c]);
  }
}

// ESPnet relative positional table (embedding.py:224-254): row m <-> relative position r = center - m,
// pe[2i] = sin(r*w_i), pe[2i+1] = cos(r*w_i), w_i = exp(-2i*ln(10000)/512)
template <typename TO>
__global__ void relpos_table_kernel(TO* __restrict__ out, int ldo, int rows, int center) {
  int m = blockIdx.x;
  if (m >= rows) return;
  float r = (float)(center - m);
  for (int i = threadIdx.x; i < D_ENC / 2; i += blockDim.x) {
    float w = expf((float)(2 * i) * -(logf(10000.0f) / (float)D_ENC));
    float a = r * w;
    out[(size_t)m * ldo + 2 * i] = from_f32<TO>(sinf(a));
    out[(size_t)m * ldo + 2 * i + 1] = from_f32<TO>(cosf(a));
  }
}

// F.normalize(embedding, dim=1) (eps 1e-12) -> [B,192]
__global__ void l2norm_kernel(const float* __restrict__ x, float* __restrict__ y, int C) {
  __shared__ float red[32];
  int b = blockIdx.x;
  float s = 0.f;
  for (int c = threadIdx.x; c < C; c += blockDim.x) s += x[(size_t)b * C + c] * x[(size_t)b * C + c];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
    t = warp_sum(t);
    if (threadIdx.x == 0) red[0] = t;
  }
  __syncthreads();
  float n = fmaxf(sqrtf(red[0]), 1e-12f);
  for (int c = threadIdx.x; c < C; c += blockDim.x) y[(size_t)b * C + c] = x[(size_t)b * C + c] / n;
}

// SinusoidalPosEmb(320), scale 1000 (matcha decoder.py:14-29): [B] -> [B,320]
__global__ void time_sincos_kernel(const float* __restrict__ t, float* __restrict__ out) {
  int b = blockIdx.x;
  const int half = 160;
  float k = logf(10000.0f) / (float)(half - 1);
  for (int i = threadIdx.x; i < half; i += blockDim.x) {
    float e = expf((float)i * -k);
    float a = 1000.f * t[b] * e;
    out[(size_t)b * 320 + i] = sinf(a);
    out[(size_t)b * 320 + half + i] = cosf(a);
  }
}

// Build the estimator input [x | mu | spks | cond] (320 ch) for the 2B sequences of the CFG batch
// (flow_matching.py:103-108: branch 1 keeps x and t, zeroes mu/spks/cond).  state/mu/cond live in the B-sequence
// geometry; the output in the 2B-sequence geometry.
template <typename TO>
__global__ void cfg_pack_kernel(const float* __restrict__ x, const float* __restrict__ mu, const float* __restrict__ cond,
                                const float* __restrict__ spks /*[B][80]*/, const int* __restrict__ start1, const int* __restrict__ start2,
                                const int* __restrict__ len, int B, TO* __restrict__ out, int ldo) {
  int b2 = blockIdx.y;
  int b = b2 % B;
  bool uncond = b2 >= B;
  int L = len[b];
  for (int t = blockIdx.x; t < L; t += gridDim.x) {
    size_t r1 = (size_t)(start1[b] + t) * N_MEL;
    TO* o = out + (size_t)(start2[b2] + t) * ldo;
    for (int c = threadIdx.x; c < N_MEL; c += blockDim.x) {
      o[c] = from_f32<TO>(x[r1 + c]);
      o[N_MEL + c] = from_f32<TO>(uncond ? 0.f : mu[r1 + c]);
      o[2 * N_MEL + c] = from_f32<TO>(uncond ? 0.f : spks[(size_t)b * N_MEL + c]);
      o[3 * N_MEL + c] = from_f32<TO>(uncond ? 0.f : cond[r1 + c]);
    }
  }
}

// x += dt * ((1+w) * v_cond - w * v_uncond)   (flow_matching.py:116-119)
__global__ void cfg_euler_kernel(float* __restrict__ x, const float* __restrict__ v, int ldv, const int* __restrict__ start1,
                                 const int* __restrict__ start2, const int* __restrict__ len, int B, float dt, float w) {
  int b = blockIdx.y;
  int L = len[b];
  for (int t = blockIdx.x; t < L; t += gridDim.x) {
    size_t r1 = (size_t)(start1[b] + t) * N_MEL;
    const float* vc = v + (size_t)(start2[b] + t) * ldv;
    const float* vu = v + (size_t)(start2[B + b] + t) * ldv;
    for (int c = threadIdx.x; c < N_MEL; c += blockDim.x) x[r1 + c] = x[r1 + c] + dt * ((1.0f + w) * vc[c] - w * vu[c]);
  }
}

// generic estimator entry: dense x/mu/cond [sum T,80] + spks [B,80] -> packed 320-channel operand
template <typename TO>
__global__ void est_pack_kernel(const float* __restrict__ x, const float* __restrict__ mu, const float* __restrict__ cond,
                                const float* __restrict__ spks, const int* __restrict__ off, const int* __restrict__ start,
                                const int* __restrict__ len, TO* __restrict__ out, int ldo) {
  int b = blockIdx.y;
  int L = len[b];
  for (int t = blockIdx.x; t < L; t += gridDim.x) {
    size_t r = (size_t)(off[b] + t) * N_MEL;
    TO* o = out + (size_t)(start[b] + t) * ldo;
    for (int c = threadIdx.x; c < N_MEL; c += blockDim.x) {
      o[c] = from_f32<TO>(x[r + c]);
      o[N_MEL + c] = from_f32<TO>(mu[r + c]);
      o[2 * N_MEL + c] = from_f32<TO>(spks[(size_t)b * N_MEL + c]);
      o[3 * N_MEL + c] = from_f32<TO>(cond[r + c]);
    }
  }
}

__global__ void noise_init_kernel(const float* __restrict__ noise, int noise_T, const int* __restrict__ start, const int* __restrict__ len,
                                  float* __restrict__ x) {
  int b = blockIdx.y;
  int L = len[b];
  for (int t = blockIdx.x; t < L; t += gridDim.x)
    for (int c = threadIdx.x; c < N_MEL; c += blockDim.x) x[(size_t)(start[b] + t) * N_MEL + c] = noise[(size_t)t * N_MEL + c];
}

int* upload(cvk_ctx* ctx, const std::vector<int>& v, cudaStream_t st) {
  int* d = (int*)ctx->arena.alloc(sizeof(int) * (v.size() ? v.size() : 1));
  if (!v.empty()) CVK_CHECK_CUDA(cudaMemcpyAsync(d, v.data(), sizeof(int) * v.size(), cudaMemcpyHostToDevice, st));
  return d;
}
std::vector<int> prefix(const int* lens, int B) {
  std::vector<int> off(B);
  int a = 0;
  for (int b = 0; b < B; ++b) { off[b] = a; a += lens[b]; }
  return off;
}

// ================================================================================================ encoder
void embed_apply(cvk_ctx* ctx, cudaStream_t st, const EmbedW& e, const Mat& in, const Seqs& s, const Mat& out_f32) {
  Mat tmp = arena_mat(ctx, DT_F32, s.R, D_ENC);
  Epilogue ep;
  ep.row2seq = s.d_row2seq;
  ep.out = tmp;
  conv_gemm(ctx, st, in, e.lin, ep);
  layernorm(ctx, st, tmp, e.ln_g, e.ln_b, 1e-5f, ACT_NONE, sqrtf((float)D_ENC), s.d_row2seq, out_f32);
}

void enc_layer(cvk_ctx* ctx, cudaStream_t st, const EncLayerW& l, const Seqs& s, const Mat& x /*fp32 residual stream*/, const Mat& pe,
               int center, int chunk) {
  const int adt = ctx->act_dtype;
  size_t mark = ctx->arena.off;
  Mat xn = arena_mat(ctx, adt, s.R, D_ENC);
  layernorm(ctx, st, x, l.ln1_g, l.ln1_b, 1e-12f, ACT_NONE, 1.f, s.d_row2seq, xn);
  Mat qkv = arena_mat(ctx, adt, s.R, 3 * D_ENC);
  {
    Epilogue e;
    e.row2seq = s.d_row2seq;
    e.out = qkv;
    conv_gemm(ctx, st, xn, l.qkv, e);
  }
  Mat p = arena_mat(ctx, adt, pe.rows, D_ENC);
  {
    Epilogue e;
    e.out = p;
    conv_gemm(ctx, st, pe, l.pos, e);
  }
  Mat att = arena_mat(ctx, adt, s.R, D_ENC);
  relpos_attention_fwd(ctx, st, qkv.slice(0, D_ENC), qkv.slice(D_ENC, D_ENC), qkv.slice(2 * D_ENC, D_ENC), p, center, l.bias_u, l.bias_v,
                       s, H_ENC, chunk, 1.0f / sqrtf(64.f), att);
  {
    Epilogue e;
    e.resid = x;
    e.row2seq = s.d_row2seq;
    e.out = x;
    conv_gemm(ctx, st, att, l.out, e);
  }
  layernorm(ctx, st, x, l.ln2_g, l.ln2_b, 1e-12f, ACT_NONE, 1.f, s.d_row2seq, xn);
  Mat ff = arena_mat(ctx, adt, s.R, FF_ENC);
  {
    Epilogue e;
    e.act1 = ACT_SILU;
    e.row2seq = s.d_row2seq;
    e.out = ff;
    conv_gemm(ctx, st, xn, l.w1, e);
  }
  {
    Epilogue e;
    e.resid = x;
    e.row2seq = s.d_row2seq;
    e.out = x;
    conv_gemm(ctx, st, ff, l.w2, e);
  }
  ctx->arena.off = mark;
}

Mat make_pe(cvk_ctx* ctx, cudaStream_t st, int max_len, int* center) {
  int rows = 2 * max_len - 1;
  Mat pe = arena_mat(ctx, ctx->act_dtype, round_up(rows, 128), D_ENC);
  zero_mat(ctx, st, pe);
  *center = max_len - 1;
  if (pe.dtype == DT_F32) relpos_table_kernel<float><<<rows, 128, 0, st>>>(pe.f32(), pe.ld, rows, *center);
  else relpos_table_kernel<bf16><<<rows, 128, 0, st>>>(pe.b16(), pe.ld, rows, *center);
  ctx->launches++;
  CVK_LAUNCH_CHECK();
  return pe;
}

// tokens (dense, sum of full lens) -> encoder output h [R2, 512] fp32 in the x2 geometry s2 (returned)
Mat encoder_forward(cvk_ctx* ctx, cudaStream_t st, const int32_t* tokens, const int* lens, int B, int streaming, int context_len,
                    Seqs* s2_out) {
  FlowModel* m = ctx->flow;
  const int adt = ctx->act_dtype;
  Seqs sf = make_seqs(ctx, lens, B, 8, 1, 0, st);                                       // all tokens incl. look-ahead context
  Seqs s1 = context_len > 0 ? shrink_seqs(ctx, sf, context_len, st) : sf;                // tokens that produce output
  int* toff = upload(ctx, prefix(lens, B), st);
  Mat emb = arena_mat(ctx, adt, sf.R, D_ENC);
  zero_mat(ctx, st, emb);
  {
    int bx = sf.max_len < 512 ? sf.max_len : 512;
    if (adt == DT_F32) token_embed_kernel<float><<<dim3(bx, B), 128, 0, st>>>(tokens, toff, m->tok_emb, sf.d_start, sf.d_len, emb.f32(), emb.ld);
    else token_embed_kernel<bf16><<<dim3(bx, B), 128, 0, st>>>(tokens, toff, m->tok_emb, sf.d_start, sf.d_len, emb.b16(), emb.ld);
    ctx->launches++;
    CVK_LAUNCH_CHECK();
  }
  // embed: Linear + LN + sqrt(d) on every token row (context rows are embedded too, upsample_encoder.py:282-284)
  Mat h0 = arena_mat(ctx, DT_F32, sf.R, D_ENC);
  embed_apply(ctx, st, m->embed, emb, sf, h0);
  // PreLookaheadLayer (:82-103): conv k4 looking right (zero pad or the context rows), leaky_relu, causal conv k3, + input
  Mat h0a = h0;
  if (adt != DT_F32) {
    h0a = arena_mat(ctx, adt, sf.R, D_ENC);
    convert_mat(ctx, st, h0, h0a);
  }
  Mat c1 = arena_mat(ctx, adt, sf.R, D_ENC);
  {
    Epilogue e;
    e.act1 = ACT_LRELU;
    e.act1_param = 0.01f;
    e.row2seq = s1.d_row2seq;
    e.out = c1;
    conv_gemm(ctx, st, h0a, m->pre1, e);
  }
  Mat x = arena_mat(ctx, DT_F32, sf.R, D_ENC);
  {
    Epilogue e;
    e.resid = h0;
    e.row2seq = s1.d_row2seq;   // rows of the context are dropped here (masked to zero)
    e.out = x;
    conv_gemm(ctx, st, c1, m->pre2, e);
  }
  int center = 0;
  Mat pe = make_pe(ctx, st, s1.max_len, &center);
  for (auto& l : m->enc) enc_layer(ctx, st, l, s1, x, pe, center, streaming ? CHUNK_TOK : 0);
  // nearest x2 + conv k5 (polyphase): [R, 2*512] == [2R, 512]
  Mat xa = x;
  if (adt != DT_F32) {
    xa = arena_mat(ctx, adt, sf.R, D_ENC);
    convert_mat(ctx, st, x, xa);
  }
  Seqs s2 = scale_seqs(ctx, s1, 2, 0, st);
  Mat up(ctx->arena.alloc((size_t)s2.R * D_ENC * (adt == DT_F32 ? 4 : 2)), adt, s1.R, 2 * D_ENC, 2 * D_ENC);
  {
    Epilogue e;
    e.row2seq = s1.d_row2seq;
    e.out = up;
    conv_gemm(ctx, st, xa, m->up_conv, e);
  }
  Mat up2(up.p, adt, s2.R, D_ENC, D_ENC);
  Mat y = arena_mat(ctx, DT_F32, s2.R, D_ENC);
  embed_apply(ctx, st, m->up_embed, up2, s2, y);
  Mat pe2 = make_pe(ctx, st, s2.max_len, &center);
  for (auto& l : m->enc_up) enc_layer(ctx, st, l, s2, y, pe2, center, streaming ? 2 * CHUNK_TOK : 0);
  Mat h = arena_mat(ctx, DT_F32, s2.R, D_ENC);
  layernorm(ctx, st, y, m->after_g, m->after_b, 1e-5f, ACT_NONE, 1.f, s2.d_row2seq, h);
  *s2_out = s2;
  return h;
}

// ================================================================================================ estimator
struct EstBuffers {
  Mat x;        // fp32 [R,256] residual stream
  Mat xa;       // act  [R,256]
  Mat cat;      // act  [R,512]  (x | skip)
  Mat c;        // fp32 [R,256]  conv pre-LN
  Mat h1;       // act  [R,256]
  Mat h2;       // fp32 [R,256]
  Mat xn;       // act  [R,256]
  Mat qkv;      // act  [R,1536]
  Mat att;      // act  [R,512]
  Mat ff;       // act  [R,1024]
  Mat temb_all; // fp32 [B2, 14*256]
};

// ---- incremental (cached) estimator call: state of ONE Euler step of one streaming session ------------------------------
// Block-causal attention (key j visible from query i iff j < (i/50+1)*50, utils/mask.py:127-158) and causal convolutions
// (flow/decoder.py:25-62: left padding k-1) make every frame of a COMPLETE 50-frame chunk independent of later frames, so a
// chunk boundary is a valid cut: per Euler step, per transformer block the K/V rows of all earlier frames, and per causal
// convolution the last two input rows, are all a later call needs.  The reference recomputes the prefix instead
// (cli/model.py:346-363).
struct EstInc {
  void* kv = nullptr;        // [n_tblocks][kv_rows][kv_width] act dtype: K | V rows, sequence b's from row kg.d_kstart[b]
  void* conv = nullptr;      // [n_convs][n_states][tail_rows][conv_c] act dtype, sequence b's tail at state cidx[b]
  int kv_width = 1024, tail_rows = 2, conv_c = 512;
  int kv_rows = 0, n_states = 0;
  int tb_idx = 0, conv_idx = 0;
  KvGeom kg;
  const int* d_cidx = nullptr;
};

template <typename T>
__global__ void conv_state_kernel(T* __restrict__ x, int ld, int C, const int* __restrict__ start, const int* __restrict__ len, T* __restrict__ state,
                                  int tail, int cstride, const int* __restrict__ cidx) {
  // gap rows start-tail .. start-1 <- saved tail of the previous chunk; saved tail <- last `tail` rows of this chunk (chunks are at
  // least 50 rows, so the two row ranges never overlap)
  const int b = blockIdx.x, r = blockIdx.y;
  T* srow = state + ((size_t)cidx[b] * tail + r) * cstride;
  T* gap = x + (size_t)(start[b] - tail + r) * ld;
  const T* tl = x + (size_t)(start[b] + len[b] - tail + r) * ld;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    gap[c] = srow[c];
    srow[c] = tl[c];
  }
}

// rows of a chunk's K | V columns (qkv columns [koff, koff + width)) appended to the cache of its sequence; the chunk's first row
// goes to cache row kstart[b] + qoff[b] (device memory, so that a captured launch stays valid from chunk to chunk)
template <typename T>
__global__ void kv_append_kernel(const T* __restrict__ qkv, int ld, int koff, int width, const int* __restrict__ start, const int* __restrict__ len,
                                 T* __restrict__ cache, const int* __restrict__ kstart, const int* __restrict__ qoff) {
  const int b = blockIdx.y;
  const int L = len[b], row0 = kstart[b] + qoff[b];
  for (int i = blockIdx.x; i < L; i += gridDim.x) {
    const uint4* src = reinterpret_cast<const uint4*>(qkv + (size_t)(start[b] + i) * ld + koff);
    uint4* dst = reinterpret_cast<uint4*>(cache + ((size_t)row0 + i) * width);
    for (int c = threadIdx.x; c < width * (int)sizeof(T) / 16; c += blockDim.x) dst[c] = src[c];
  }
}

// inputs of one multi-slot chunk call: sequence b (slot slot[b], frames [t_prev[b], t_prev[b] + len1[b])) gets its new rows of mu
// (mu_full, geometry start2), of the CFM noise, and of its slot's prompt conditioning (zero past pfr[b]) in geometry start1, and
// its slot's speaker row in spk_out[b]
__global__ void stream_gather_kernel(const float* __restrict__ mu_full, const int* __restrict__ start2, const float* __restrict__ noise,
                                     const float* __restrict__ prompt_feat, const float* __restrict__ spk, int cap,
                                     const int* __restrict__ geo /*t_prev[B] | pfr[B] | slot[B]*/, int B, const int* __restrict__ start1,
                                     const int* __restrict__ len1, float* __restrict__ mu, float* __restrict__ cond, float* __restrict__ x,
                                     float* __restrict__ spk_out) {
  const int b = blockIdx.y;
  const int t_prev = geo[b], pfr = geo[B + b], slot = geo[2 * B + b], L = len1[b];
  if (blockIdx.x == 0)
    for (int c = threadIdx.x; c < N_MEL; c += blockDim.x) spk_out[(size_t)b * N_MEL + c] = spk[(size_t)slot * N_MEL + c];
  for (int t = blockIdx.x; t < L; t += gridDim.x) {
    const int g = t_prev + t;
    const size_t r1 = (size_t)(start1[b] + t) * N_MEL;
    const float* m = mu_full + (size_t)(start2[b] + g) * N_MEL;
    const float* pf = prompt_feat + ((size_t)slot * cap + g) * N_MEL;
    for (int c = threadIdx.x; c < N_MEL; c += blockDim.x) {
      mu[r1 + c] = m[c];
      x[r1 + c] = noise[(size_t)g * N_MEL + c];
      cond[r1 + c] = g < pfr ? pf[c] : 0.f;
    }
  }
}

// the two rows a causal k=3 convolution reads in front of the chunk (call right before the convolution that consumes `in`)
void conv_state(cvk_ctx* ctx, cudaStream_t st, EstInc* inc, const Mat& in, const Seqs& s) {
  if (!inc) return;
  CVK_REQUIRE(in.cols <= inc->conv_c && s.B <= inc->n_states, "conv_state: unexpected operand");
  const size_t es = in.esize();
  char* state = (char*)inc->conv + (size_t)inc->conv_idx * inc->n_states * inc->tail_rows * inc->conv_c * es;
  ++inc->conv_idx;
  if (in.dtype == DT_F32)
    conv_state_kernel<float><<<dim3(s.B, inc->tail_rows), 128, 0, st>>>(in.f32(), in.ld, in.cols, s.d_start, s.d_len, (float*)state, inc->tail_rows, inc->conv_c,
                                                                        inc->d_cidx);
  else
    conv_state_kernel<bf16><<<dim3(s.B, inc->tail_rows), 128, 0, st>>>(in.b16(), in.ld, in.cols, s.d_start, s.d_len, (bf16*)state, inc->tail_rows, inc->conv_c,
                                                                       inc->d_cidx);
  ctx->launches++;
  CVK_LAUNCH_CHECK();
}

// append the chunk's K | V rows (columns [koff, koff + kv_width) of qkv) to the cache of the next block and return that cache
Mat kv_cache_append(cvk_ctx* ctx, cudaStream_t st, EstInc* inc, const Mat& qkv, int koff, const Seqs& s) {
  const size_t es = qkv.esize();
  const int crow = inc->kv_rows;
  Mat cache((char*)inc->kv + (size_t)inc->tb_idx * crow * inc->kv_width * es, qkv.dtype, crow, inc->kv_width, inc->kv_width);
  ++inc->tb_idx;
  int bx = s.max_len < 256 ? s.max_len : 256;
  if (qkv.dtype == DT_F32)
    kv_append_kernel<float><<<dim3(bx, s.B), 128, 0, st>>>(qkv.f32(), qkv.ld, koff, inc->kv_width, s.d_start, s.d_len, cache.f32(), inc->kg.d_kstart,
                                                           inc->kg.d_qoff);
  else
    kv_append_kernel<bf16><<<dim3(bx, s.B), 128, 0, st>>>(qkv.b16(), qkv.ld, koff, inc->kv_width, s.d_start, s.d_len, cache.b16(), inc->kg.d_kstart,
                                                          inc->kg.d_qoff);
  ctx->launches++;
  CVK_LAUNCH_CHECK();
  return cache;
}

void tblock(cvk_ctx* ctx, cudaStream_t st, const TBlockW& t, const Seqs& s, EstBuffers& b, int chunk, const Mat* out2, EstInc* inc = nullptr) {
  layernorm(ctx, st, b.x, t.ln1_g, t.ln1_b, 1e-5f, ACT_NONE, 1.f, s.d_row2seq, b.xn);
  {
    Epilogue e;
    e.row2seq = s.d_row2seq;
    e.out = b.qkv;
    conv_gemm(ctx, st, b.xn, t.qkv, e);
  }
  if (inc) {
    Mat cache = kv_cache_append(ctx, st, inc, b.qkv, 512, s);
    attention_fwd(ctx, st, b.qkv.slice(0, 512), cache.slice(0, 512), cache.slice(512, 512), s, H_EST, chunk, 0.125f, b.att, 1, &inc->kg);
  } else
  attention_fwd(ctx, st, b.qkv.slice(0, 512), b.qkv.slice(512, 512), b.qkv.slice(1024, 512), s, H_EST, chunk, 0.125f, b.att);
  {
    Epilogue e;
    e.resid = b.x;
    e.row2seq = s.d_row2seq;
    e.out = b.x;
    conv_gemm(ctx, st, b.att, t.out, e);
  }
  layernorm(ctx, st, b.x, t.ln3_g, t.ln3_b, 1e-5f, ACT_NONE, 1.f, s.d_row2seq, b.xn);
  {
    Epilogue e;
    e.act1 = ACT_GELU;
    e.row2seq = s.d_row2seq;
    e.out = b.ff;
    conv_gemm(ctx, st, b.xn, t.ff1, e);
  }
  {
    Epilogue e;
    e.resid = b.x;
    e.row2seq = s.d_row2seq;
    e.out = b.x;
    if (out2) {
      e.act2 = ACT_NONE;
      e.out2 = *out2;
    }
    conv_gemm(ctx, st, b.ff, t.ff2, e);
  }
}

// resnet (matcha decoder.py:55-61 with CausalBlock1D) + n transformer blocks.  `in` = act operand [R, Cin];
// the stage's output residual stream ends in b.x (fp32) and, as an activation operand, in *out_act.
void stage_forward(cvk_ctx* ctx, cudaStream_t st, const StageW& w, int stage_idx, const Seqs& s, const Mat& in, EstBuffers& b, int chunk,
                   const Mat& out_act, EstInc* inc = nullptr) {
  const float* tvec = b.temb_all.f32() + (size_t)stage_idx * C_EST;
  conv_state(ctx, st, inc, in, s);
  {
    Epilogue e;
    e.row2seq = s.d_row2seq;
    e.out = b.c;
    conv_gemm(ctx, st, in, w.rn.c1, e);
  }
  layernorm(ctx, st, b.c, w.rn.ln1_g, w.rn.ln1_b, 1e-5f, ACT_MISH, 1.f, s.d_row2seq, b.h1, tvec, b.temb_all.ld);
  conv_state(ctx, st, inc, b.h1, s);
  {
    Epilogue e;
    e.row2seq = s.d_row2seq;
    e.out = b.c;
    conv_gemm(ctx, st, b.h1, w.rn.c2, e);
  }
  layernorm(ctx, st, b.c, w.rn.ln2_g, w.rn.ln2_b, 1e-5f, ACT_MISH, 1.f, s.d_row2seq, b.h2);
  {
    Epilogue e;
    e.resid = b.h2;
    e.row2seq = s.d_row2seq;
    e.out = b.x;
    conv_gemm(ctx, st, in, w.rn.res, e);
  }
  for (size_t j = 0; j < w.tb.size(); ++j) tblock(ctx, st, w.tb[j], s, b, chunk, j + 1 == w.tb.size() ? &out_act : nullptr, inc);
}

// in0: act [R,320] packed input; t: [B2] device; out: fp32 [R,80] (ld 80)
void estimator_forward(cvk_ctx* ctx, cudaStream_t st, const Seqs& s, const Mat& in0, const float* t_dev, int streaming, const Mat& out,
                       EstInc* inc = nullptr) {
  FlowModel* m = ctx->flow;
  const int adt = ctx->act_dtype;
  const int chunk = streaming ? 2 * CHUNK_TOK : 0;
  size_t mark = ctx->arena.off;
  EstBuffers b;
  b.x = arena_mat(ctx, DT_F32, s.R, C_EST);
  b.xa = arena_mat(ctx, adt, s.R, C_EST);
  b.cat = arena_mat(ctx, adt, s.R, 2 * C_EST);
  b.c = arena_mat(ctx, DT_F32, s.R, C_EST);
  b.h1 = arena_mat(ctx, adt, s.R, C_EST);
  b.h2 = arena_mat(ctx, DT_F32, s.R, C_EST);
  b.xn = arena_mat(ctx, adt, s.R, C_EST);
  b.qkv = arena_mat(ctx, adt, s.R, 3 * 512);
  b.att = arena_mat(ctx, adt, s.R, 512);
  b.ff = arena_mat(ctx, adt, s.R, 4 * C_EST);
  // time embedding -> all 14 per-stage projections at once
  const int nst = (int)m->stages.size();
  Mat sc = arena_mat(ctx, DT_F32, s.B, 320);
  time_sincos_kernel<<<s.B, 160, 0, st>>>(t_dev, sc.f32());
  ctx->launches++;
  CVK_LAUNCH_CHECK();
  Mat te1 = arena_mat(ctx, DT_F32, s.B, TEMB), te2 = arena_mat(ctx, DT_F32, s.B, TEMB), te3 = arena_mat(ctx, DT_F32, s.B, TEMB);
  {
    Epilogue e;
    e.act1 = ACT_SILU;
    e.out = te1;
    conv_gemm_simt(ctx, st, sc, m->t1, e);
  }
  {
    Epilogue e;
    e.out = te2;
    e.act2 = ACT_MISH;       // ResnetBlock1D.mlp = Sequential(Mish, Linear)
    e.out2 = te3;
    conv_gemm_simt(ctx, st, te1, m->t2, e);
  }
  b.temb_all = arena_mat(ctx, DT_F32, s.B, nst * C_EST);
  {
    Epilogue e;
    e.out = b.temb_all;
    conv_gemm_simt(ctx, st, te3, m->tmlp_all, e);
  }
  // down stage: output -> skip half of `cat`
  stage_forward(ctx, st, m->stages[0], 0, s, in0, b, chunk, b.cat.slice(C_EST, C_EST), inc);
  conv_state(ctx, st, inc, b.cat.slice(C_EST, C_EST), s);
  {
    Epilogue e;      // down_blocks.0.2 causal conv on the skip tensor
    e.row2seq = s.d_row2seq;
    e.out = b.xa;
    conv_gemm(ctx, st, b.cat.slice(C_EST, C_EST), m->down_conv, e);
  }
  for (int i = 0; i < m->num_mid; ++i) {
    bool last = i + 1 == m->num_mid;
    stage_forward(ctx, st, m->stages[1 + i], 1 + i, s, b.xa, b, chunk, last ? b.cat.slice(0, C_EST) : b.xa, inc);
  }
  if (m->num_mid == 0) convert_mat(ctx, st, b.xa, b.cat.slice(0, C_EST));
  stage_forward(ctx, st, m->stages[nst - 1], nst - 1, s, b.cat, b, chunk, b.xa, inc);
  conv_state(ctx, st, inc, b.xa, s);
  {
    Epilogue e;      // up_blocks.0.2
    e.row2seq = s.d_row2seq;
    e.out = b.h1;
    conv_gemm(ctx, st, b.xa, m->up_conv2, e);
  }
  conv_state(ctx, st, inc, b.h1, s);
  {
    Epilogue e;      // final CausalBlock1D
    e.row2seq = s.d_row2seq;
    e.out = b.c;
    conv_gemm(ctx, st, b.h1, m->final_conv, e);
  }
  layernorm(ctx, st, b.c, m->final_g, m->final_b, 1e-5f, ACT_MISH, 1.f, s.d_row2seq, b.xa);
  {
    Epilogue e;
    e.row2seq = s.d_row2seq;
    e.out = out;
    conv_gemm(ctx, st, b.xa, m->final_proj, e);
  }
  ctx->arena.off = mark;
}

// mu, cond, x: fp32 [R1,80] (ld 80) in geometry s1; spks [B,80].  Runs n Euler steps in place on x.
void dit_estimator_forward(cvk_ctx* ctx, cudaStream_t st, const Seqs& s, const Mat& in0, const float* t_dev, int streaming, const Mat& out,
                           EstInc* inc);

// `dit`: 0 = CosyVoice2 causal U-Net estimator, 1 = CosyVoice3 DiT (32 gap rows: its causal position convolution looks 30 rows back)
void cfm_solve_packed(cvk_ctx* ctx, cudaStream_t st, const Seqs& s1, const int* lens, const Mat& mu, const Mat& cond, const float* spks,
                      const Mat& x, int n_timesteps, float cfg_rate, int streaming, int dit = 0, cvk_flow_stream* fs = nullptr) {
  const int adt = ctx->act_dtype;
  const int B = s1.B;
  std::vector<int> lens2(2 * B);
  for (int b = 0; b < 2 * B; ++b) lens2[b] = lens[b % B];
  Seqs s2 = make_seqs(ctx, lens2.data(), 2 * B, dit ? 32 : 8, 1, 0, st);
  Mat in0 = arena_mat(ctx, adt, s2.R, 320);
  zero_mat(ctx, st, in0);
  Mat v = arena_mat(ctx, DT_F32, s2.R, N_MEL, N_MEL);
  float* t_dev = (float*)ctx->arena.alloc(sizeof(float) * 2 * B * (n_timesteps + 1));
  // t_span = 1 - cos(linspace(0,1,n+1) * pi/2), float32 like torch (flow_matching.py:224-226)
  std::vector<float> tspan(n_timesteps + 1);
  for (int i = 0; i <= n_timesteps; ++i) {
    float lin = (float)i / (float)n_timesteps;
    if (i == n_timesteps) lin = 1.0f;
    tspan[i] = 1.0f - cosf(lin * 0.5f * 3.14159265358979323846f);
  }
  // per-step t values replicated for the 2B sequences
  std::vector<float> tall((size_t)(n_timesteps + 1) * 2 * B);
  float t = tspan[0], dt = tspan[1] - tspan[0];
  std::vector<float> dts(n_timesteps);
  for (int step = 1; step <= n_timesteps; ++step) {
    for (int b = 0; b < 2 * B; ++b) tall[(size_t)(step - 1) * 2 * B + b] = t;
    dts[step - 1] = dt;
    t = t + dt;
    if (step < n_timesteps) dt = tspan[step + 1] - t;
  }
  CVK_CHECK_CUDA(cudaMemcpyAsync(t_dev, tall.data(), sizeof(float) * (size_t)n_timesteps * 2 * B, cudaMemcpyHostToDevice, st));
  int bx = s1.max_len < 1024 ? s1.max_len : 1024;
  for (int step = 0; step < n_timesteps; ++step) {
    if (adt == DT_F32)
      cfg_pack_kernel<float><<<dim3(bx, 2 * B), 96, 0, st>>>(x.f32(), mu.f32(), cond.f32(), spks, s1.d_start, s2.d_start, s1.d_len, B, in0.f32(), in0.ld);
    else
      cfg_pack_kernel<bf16><<<dim3(bx, 2 * B), 96, 0, st>>>(x.f32(), mu.f32(), cond.f32(), spks, s1.d_start, s2.d_start, s1.d_len, B, in0.b16(), in0.ld);
    ctx->launches++;
    CVK_LAUNCH_CHECK();
    if (fs) {
      EstInc inc;
      inc.kv = (char*)fs->kv + (size_t)step * fs->kv_step_bytes;
      inc.conv = (char*)fs->conv + (size_t)step * fs->conv_step_bytes;
      inc.kv_rows = 2 * fs->n_slots * fs->cap + 64;
      inc.n_states = 2 * fs->n_slots;
      inc.kg = fs->kg;
      inc.d_cidx = fs->d_cidx;
      inc.kv_width = fs->kv_width; inc.tail_rows = fs->tail_rows; inc.conv_c = fs->conv_c;
      if (dit) dit_estimator_forward(ctx, st, s2, in0, t_dev + (size_t)step * 2 * B, streaming, v, &inc);
      else estimator_forward(ctx, st, s2, in0, t_dev + (size_t)step * 2 * B, streaming, v, &inc);
      CVK_REQUIRE(inc.tb_idx == fs->n_tb && inc.conv_idx == fs->n_conv, "flow stream: cache slots do not match the estimator");
    } else if (dit) dit_estimator_forward(ctx, st, s2, in0, t_dev + (size_t)step * 2 * B, streaming, v, nullptr);
    else estimator_forward(ctx, st, s2, in0, t_dev + (size_t)step * 2 * B, streaming, v);
    cfg_euler_kernel<<<dim3(bx, B), 96, 0, st>>>(x.f32(), v.f32(), v.ld, s1.d_start, s2.d_start, s1.d_len, B, dts[step], cfg_rate);
    ctx->launches++;
    CVK_LAUNCH_CHECK();
  }
}


// ================================================================================================ CosyVoice3 DiT estimator
// cosyvoice/flow/DiT/dit.py:104-176 + modules.py (TimestepEmbedding :606-616, CausalConvPositionEmbedding :115-145, DiTBlock
// :500-533, AdaLayerNormZero :230-248, AdaLayerNormZero_Final :251-264, AttnProcessor :349-411), cosyvoice3.yaml: dim 1024,
// depth 22, 16 heads x 64, ff_mult 2, static chunk 50.  Same packed time-major layout as the U-Net estimator: the CFG pair is
// 2B sequences; AdaLN modulation vectors are per-SEQUENCE rows of one [2B, depth*6144 + 2048] matrix produced by ONE GEMM per
// estimator call (the time embedding is shared by all blocks); the grouped causal position convolution (k31, 16 groups) is 16
// conv-GEMMs on 64-column slices; the rotary embedding touches the first 64 channels of q and k only (x_transformers partial
// rotary on the un-split projection, modules.py:368-373).
constexpr int DIT_D = 1024, DIT_H = 16, DIT_FF = 2048, DIT_GROUPS = 16, DIT_CK = 31;

struct DitBlockW {
  ConvW qkv, out, ff1, ff2;
};
}  // namespace

struct DitModel {
  int depth = 22;
  float* tok_emb = nullptr;        // [6561][80]
  ConvW spk_affine, pre1, pre2;    // 192 -> 80; PreLookaheadLayer(80, 1024, 3)
  ConvW t1, t2;                    // time MLP 256 -> 1024 -> 1024
  ConvW in_proj;                   // 320 -> 1024, input columns permuted to the [x | mu | spks | cond] packing of cfg_pack_kernel
  std::vector<ConvW> pos1, pos2;   // 16 groups each: [64][31][64]
  ConvW mod_all;                   // [depth*6144 + 2048][1024]: every attn_norm.linear, then norm_out.linear
  std::vector<DitBlockW> blocks;
  ConvW proj_out;                  // 1024 -> 80
};

namespace {

// modules.py:71-84 with dim 256, scale 1000: emb = exp(-i * ln(1e4)/(127)), [sin | cos]
__global__ void dit_time_sincos_kernel(const float* __restrict__ t, float* __restrict__ out) {
  const int b = blockIdx.x, half = 128;
  const float k = logf(10000.0f) / (float)(half - 1);
  for (int i = threadIdx.x; i < half; i += blockDim.x) {
    const float a = 1000.f * t[b] * expf((float)i * -k);
    out[(size_t)b * 256 + i] = sinf(a);
    out[(size_t)b * 256 + half + i] = cosf(a);
  }
}

// in_proj weight [1024][320] with reference column order [x | cond | mu | spks] (dit.py:91-97) -> [x | mu | spks | cond]
__global__ void dit_permute_inproj_kernel(const float* __restrict__ w, float* __restrict__ o, int N) {
  const size_t total = (size_t)N * 320;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int n = (int)(i / 320), c = (int)(i % 320);
    const int blk = c / 80, j = c % 80;                  // destination block: 0 x, 1 mu, 2 spks, 3 cond
    const int src = blk == 0 ? j : (blk == 1 ? 160 + j : (blk == 2 ? 240 + j : 80 + j));
    o[i] = w[(size_t)n * 320 + src];
  }
}

// LayerNorm(1024, no affine, eps 1e-6) followed by the per-sequence modulation  y = norm * (1 + scale[seq]) + shift[seq]
// (modules.py:245-247, 262-263, 527); one warp per row, the row in registers (8 x float4 per lane)
template <typename TO>
__global__ void layernorm_mod_kernel(const float* __restrict__ x, int ldx, int rows, const int* __restrict__ row2seq,
                                     const float* __restrict__ scale, const float* __restrict__ shift, int mod_ld, TO* __restrict__ out, int ldo) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (row >= rows) return;
  const int seq = row2seq[row];
  TO* op = out + (size_t)row * ldo;
  float v[32];
  if (seq < 0) {
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = 0.f;
  } else {
    const float* xp = x + (size_t)row * ldx;
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 a = *reinterpret_cast<const float4*>(xp + j * 128 + lane * 4);
      v[4 * j] = a.x; v[4 * j + 1] = a.y; v[4 * j + 2] = a.z; v[4 * j + 3] = a.w;
      s += (a.x + a.y) + (a.z + a.w);
    }
    const float mean = warp_sum(s) * (1.f / DIT_D);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      v[i] -= mean;
      q = fmaf(v[i], v[i], q);
    }
    const float rstd = rsqrtf(warp_sum(q) * (1.f / DIT_D) + 1e-6f);
    const float* sc = scale + (size_t)seq * mod_ld;
    const float* sh = shift + (size_t)seq * mod_ld;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 a = *reinterpret_cast<const float4*>(sc + j * 128 + lane * 4);
      const float4 b = *reinterpret_cast<const float4*>(sh + j * 128 + lane * 4);
      v[4 * j] = fmaf(v[4 * j] * rstd, 1.f + a.x, b.x);
      v[4 * j + 1] = fmaf(v[4 * j + 1] * rstd, 1.f + a.y, b.y);
      v[4 * j + 2] = fmaf(v[4 * j + 2] * rstd, 1.f + a.z, b.z);
      v[4 * j + 3] = fmaf(v[4 * j + 3] * rstd, 1.f + a.w, b.w);
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    TO* o = op + j * 128 + lane * 4;
    o[0] = from_f32<TO>(v[4 * j]); o[1] = from_f32<TO>(v[4 * j + 1]); o[2] = from_f32<TO>(v[4 * j + 2]); o[3] = from_f32<TO>(v[4 * j + 3]);
  }
}

// x[r, :] += gate[seq(r), :] * o[r, :]   (modules.py:526, 530; gap rows stay zero because o is masked there)
__global__ void dit_gate_add_kernel(float* __restrict__ x, int ldx, const float* __restrict__ o, int ldo, int rows,
                                    const int* __restrict__ row2seq, const float* __restrict__ gate, int gate_ld) {
  const size_t total = (size_t)rows * (DIT_D / 4);
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / (DIT_D / 4)), c = (int)(i % (DIT_D / 4)) * 4;
    const int seq = row2seq[r];
    if (seq < 0) continue;
    const float4 g = *reinterpret_cast<const float4*>(gate + (size_t)seq * gate_ld + c);
    const float4 a = *reinterpret_cast<const float4*>(o + (size_t)r * ldo + c);
    float4 v = *reinterpret_cast<float4*>(x + (size_t)r * ldx + c);
    v.x = fmaf(g.x, a.x, v.x); v.y = fmaf(g.y, a.y, v.y); v.z = fmaf(g.z, a.z, v.z); v.w = fmaf(g.w, a.w, v.w);
    *reinterpret_cast<float4*>(x + (size_t)r * ldx + c) = v;
  }
}

// x_transformers partial rotary on the first 64 channels of q (columns 0..63 of the fused qkv row) and k (columns 1024..1087):
// freqs duplicated in adjacent channels, pairs (2i, 2i+1) -> (a cos - b sin, b cos + a sin), angle = position * 10000^(-2i/64)
template <typename T>
__global__ void dit_rope_kernel(T* __restrict__ qkv, int ld, const int* __restrict__ start, const int* __restrict__ len, const int* __restrict__ qoff) {
  const int b = blockIdx.y, L = len[b], p0 = qoff ? qoff[b] : 0;
  for (int t = blockIdx.x; t < L; t += gridDim.x) {
    T* row = qkv + (size_t)(start[b] + t) * ld;
    for (int e = threadIdx.x; e < 64; e += blockDim.x) {       // 32 pairs of q, 32 pairs of k
      const int which = e >> 5, i = e & 31;
      T* p = row + which * DIT_D + 2 * i;
      const float ang = (float)(p0 + t) * exp2f(-(float)(2 * i) / 64.f * 13.287712379549449f);    // log2(10000)
      const float c = cosf(ang), sn = sinf(ang);
      const float a = to_f32(p[0]), bb = to_f32(p[1]);
      p[0] = from_f32<T>(a * c - bb * sn);
      p[1] = from_f32<T>(bb * c + a * sn);
    }
  }
}

// out[2t] = out[2t+1] = in[t]  (repeat_interleave(token_mel_ratio = 2, dim=1), flow.py:393)
__global__ void repeat2_rows_kernel(const float* __restrict__ in, int ldi, const int* __restrict__ start_in, const int* __restrict__ len_in,
                                    float* __restrict__ out, int ldo, const int* __restrict__ start_out, int C) {
  const int b = blockIdx.y, L = len_in[b];
  for (int t = blockIdx.x; t < L; t += gridDim.x) {
    const float* src = in + (size_t)(start_in[b] + t) * ldi;
    float* d0 = out + (size_t)(start_out[b] + 2 * t) * ldo;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
      d0[c] = src[c];
      d0[ldo + c] = src[c];
    }
  }
}

void ln_mod(cvk_ctx* ctx, cudaStream_t st, const Mat& x, const Seqs& s, const float* scale, const float* shift, int mod_ld, const Mat& out) {
  const int blocks = ceil_div(x.rows, 8);
  if (out.dtype == DT_F32)
    layernorm_mod_kernel<float><<<blocks, 256, 0, st>>>(x.f32(), x.ld, x.rows, s.d_row2seq, scale, shift, mod_ld, out.f32(), out.ld);
  else
    layernorm_mod_kernel<bf16><<<blocks, 256, 0, st>>>(x.f32(), x.ld, x.rows, s.d_row2seq, scale, shift, mod_ld, out.b16(), out.ld);
  ctx->launches++;
  CVK_LAUNCH_CHECK();
}

void gate_add(cvk_ctx* ctx, cudaStream_t st, const Mat& x, const Mat& o, const Seqs& s, const float* gate, int gate_ld) {
  dit_gate_add_kernel<<<148 * 8, 256, 0, st>>>(x.f32(), x.ld, o.f32(), o.ld, x.rows, s.d_row2seq, gate, gate_ld);
  ctx->launches++;
  CVK_LAUNCH_CHECK();
}

// in0: act [R,320] packed [x | mu | spks | cond]; t_dev [B]; out fp32 [R,80]
void dit_estimator_forward(cvk_ctx* ctx, cudaStream_t st, const Seqs& s, const Mat& in0, const float* t_dev, int streaming, const Mat& out,
                           EstInc* inc) {
  DitModel* m = ctx->dit;
  CVK_REQUIRE(m && m->tok_emb, "flow3 stage not finalised");
  const int adt = ctx->act_dtype;
  const int chunk = streaming ? 2 * CHUNK_TOK : 0;
  const size_t mark = ctx->arena.off;
  Mat x = arena_mat(ctx, DT_F32, s.R, DIT_D), xn = arena_mat(ctx, adt, s.R, DIT_D), qkv = arena_mat(ctx, adt, s.R, 3 * DIT_D),
      att = arena_mat(ctx, adt, s.R, DIT_D), ff = arena_mat(ctx, adt, s.R, DIT_FF), o = arena_mat(ctx, DT_F32, s.R, DIT_D);
  // time embedding -> SiLU -> every modulation vector of the network in one GEMM
  Mat sc = arena_mat(ctx, DT_F32, s.B, 256), te1 = arena_mat(ctx, DT_F32, s.B, DIT_D), te = arena_mat(ctx, DT_F32, s.B, DIT_D),
      ste = arena_mat(ctx, DT_F32, s.B, DIT_D);
  dit_time_sincos_kernel<<<s.B, 128, 0, st>>>(t_dev, sc.f32());
  ctx->launches++;
  CVK_LAUNCH_CHECK();
  {
    Epilogue e;
    e.act1 = ACT_SILU;
    e.out = te1;
    conv_gemm_simt(ctx, st, sc, m->t1, e);
  }
  {
    Epilogue e;
    e.out = te;
    e.act2 = ACT_SILU;            // AdaLayerNormZero: linear(silu(emb))
    e.out2 = ste;
    conv_gemm_simt(ctx, st, te1, m->t2, e);
  }
  const int mod_ld = m->depth * 6 * DIT_D + 2 * DIT_D;
  Mat mod = arena_mat(ctx, DT_F32, s.B, mod_ld);
  {
    Epilogue e;
    e.out = mod;
    conv_gemm_simt(ctx, st, ste, m->mod_all, e);
  }
  // input embedding: proj + causal grouped position convolution (twice, Mish) + residual
  {
    Epilogue e;
    e.row2seq = s.d_row2seq;
    e.out = x;
    conv_gemm(ctx, st, in0, m->in_proj, e);
  }
  Mat xa = x;
  if (adt != DT_F32) {
    xa = xn;                      // free at this point
    convert_mat(ctx, st, x, xa);
  }
  Mat c1 = att;                   // act [R,1024], free at this point
  conv_state(ctx, st, inc, xa, s);        // streaming session: the 30 rows the k31 position convolution reads in front of the chunk
  for (int g = 0; g < DIT_GROUPS; ++g) {
    Epilogue e;
    e.act1 = ACT_MISH;
    e.row2seq = s.d_row2seq;
    e.out = c1.slice(g * 64, 64);
    conv_gemm(ctx, st, xa.slice(g * 64, 64), m->pos1[g], e);
  }
  conv_state(ctx, st, inc, c1, s);
  for (int g = 0; g < DIT_GROUPS; ++g) {
    Epilogue e;
    e.act1 = ACT_MISH;
    e.resid = x.slice(g * 64, 64);
    e.row2seq = s.d_row2seq;
    e.out = x.slice(g * 64, 64);
    conv_gemm(ctx, st, c1.slice(g * 64, 64), m->pos2[g], e);
  }
  const int bx = s.max_len < 1024 ? s.max_len : 1024;
  for (int i = 0; i < m->depth; ++i) {
    const DitBlockW& w = m->blocks[i];
    const float* mb = mod.f32() + (size_t)i * 6 * DIT_D;   // [shift_msa | scale_msa | gate_msa | shift_mlp | scale_mlp | gate_mlp]
    ln_mod(ctx, st, x, s, mb + DIT_D, mb, mod_ld, xn);
    {
      Epilogue e;
      e.row2seq = s.d_row2seq;
      e.out = qkv;
      conv_gemm(ctx, st, xn, w.qkv, e);
    }
    const int* qoff = inc ? inc->kg.d_qoff : nullptr;      // absolute position of the chunk's first row (streaming session)
    if (adt == DT_F32) dit_rope_kernel<float><<<dim3(bx, s.B), 64, 0, st>>>(qkv.f32(), qkv.ld, s.d_start, s.d_len, qoff);
    else dit_rope_kernel<bf16><<<dim3(bx, s.B), 64, 0, st>>>(qkv.b16(), qkv.ld, s.d_start, s.d_len, qoff);
    ctx->launches++;
    CVK_LAUNCH_CHECK();
    if (inc) {
      Mat cache = kv_cache_append(ctx, st, inc, qkv, DIT_D, s);
      attention_fwd(ctx, st, qkv.slice(0, DIT_D), cache.slice(0, DIT_D), cache.slice(DIT_D, DIT_D), s, DIT_H, chunk, 0.125f, att, 1, &inc->kg);
    } else
    attention_fwd(ctx, st, qkv.slice(0, DIT_D), qkv.slice(DIT_D, DIT_D), qkv.slice(2 * DIT_D, DIT_D), s, DIT_H, chunk, 0.125f, att);
    {
      Epilogue e;
      e.row2seq = s.d_row2seq;
      e.out = o;
      conv_gemm(ctx, st, att, w.out, e);
    }
    gate_add(ctx, st, x, o, s, mb + 2 * DIT_D, mod_ld);
    ln_mod(ctx, st, x, s, mb + 4 * DIT_D, mb + 3 * DIT_D, mod_ld, xn);
    {
      Epilogue e;
      e.act1 = ACT_GELU_TANH;
      e.row2seq = s.d_row2seq;
      e.out = ff;
      conv_gemm(ctx, st, xn, w.ff1, e);
    }
    {
      Epilogue e;
      e.row2seq = s.d_row2seq;
      e.out = o;
      conv_gemm(ctx, st, ff, w.ff2, e);
    }
    gate_add(ctx, st, x, o, s, mb + 5 * DIT_D, mod_ld);
  }
  const float* mf = mod.f32() + (size_t)m->depth * 6 * DIT_D;   // norm_out: [scale | shift] (modules.py:261)
  ln_mod(ctx, st, x, s, mf, mf + DIT_D, mod_ld, xn);
  {
    Epilogue e;
    e.row2seq = s.d_row2seq;
    e.out = out;
    conv_gemm(ctx, st, xn, m->proj_out, e);
  }
  ctx->arena.off = mark;
}

}  // namespace

// ================================================================================================ entry points
void flow_encoder(cvk_ctx* ctx, const int32_t* tokens, const int* lens, int B, int streaming, int context_len, float* h_out, cudaStream_t st) {
  CVK_REQUIRE(ctx->flow && ctx->flow->tok_emb, "flow stage not finalised");
  ctx->arena.reset();
  Seqs s2;
  Mat h = encoder_forward(ctx, st, tokens, lens, B, streaming, context_len, &s2);
  unpack_rows(ctx, st, h, s2, 0, h_out, D_ENC);
}

void flow_estimator(cvk_ctx* ctx, const float* x, const float* mu, const float* t, const float* spks, const float* cond, const int* lens,
                    int B, int streaming, float* out, cudaStream_t st) {
  CVK_REQUIRE(ctx->flow && ctx->flow->tok_emb, "flow stage not finalised");
  ctx->arena.reset();
  const int adt = ctx->act_dtype;
  Seqs s = make_seqs(ctx, lens, B, 8, 1, 0, st);
  Mat in0 = arena_mat(ctx, adt, s.R, 320);
  zero_mat(ctx, st, in0);
  int* off = upload(ctx, prefix(lens, B), st);
  int bx = s.max_len < 1024 ? s.max_len : 1024;
  if (adt == DT_F32) est_pack_kernel<float><<<dim3(bx, B), 96, 0, st>>>(x, mu, cond, spks, off, s.d_start, s.d_len, in0.f32(), in0.ld);
  else est_pack_kernel<bf16><<<dim3(bx, B), 96, 0, st>>>(x, mu, cond, spks, off, s.d_start, s.d_len, in0.b16(), in0.ld);
  ctx->launches++;
  CVK_LAUNCH_CHECK();
  Mat v = arena_mat(ctx, DT_F32, s.R, N_MEL, N_MEL);
  estimator_forward(ctx, st, s, in0, t, streaming, v);
  unpack_rows(ctx, st, v, s, 0, out, N_MEL);
}

void flow_cfm_solve(cvk_ctx* ctx, const float* mu, const float* spks, const float* cond, const int* lens, int B, const float* z,
                    int n_timesteps, float cfg_rate, int streaming, float* out, cudaStream_t st) {
  FlowModel* m = ctx->flow;
  CVK_REQUIRE(m && m->tok_emb, "flow stage not finalised");
  ctx->arena.reset();
  Seqs s1 = make_seqs(ctx, lens, B, 8, 1, 0, st);
  Mat mu_p = arena_mat(ctx, DT_F32, s1.R, N_MEL, N_MEL), cond_p = arena_mat(ctx, DT_F32, s1.R, N_MEL, N_MEL),
      x = arena_mat(ctx, DT_F32, s1.R, N_MEL, N_MEL);
  zero_mat(ctx, st, mu_p); zero_mat(ctx, st, cond_p); zero_mat(ctx, st, x);
  pack_rows(ctx, st, mu, N_MEL, s1, mu_p);
  pack_rows(ctx, st, cond, N_MEL, s1, cond_p);
  if (z) pack_rows(ctx, st, z, N_MEL, s1, x);
  else {
    CVK_REQUIRE(m->noise && m->noise_T >= s1.max_len, "cvk_cfm_set_noise has not been called (or the noise tensor is too short)");
    int bx = s1.max_len < 1024 ? s1.max_len : 1024;
    noise_init_kernel<<<dim3(bx, B), 96, 0, st>>>(m->noise, m->noise_T, s1.d_start, s1.d_len, x.f32());
    ctx->launches++;
    CVK_LAUNCH_CHECK();
  }
  cfm_solve_packed(ctx, st, s1, lens, mu_p, cond_p, spks, x, n_timesteps, cfg_rate, streaming);
  unpack_rows(ctx, st, x, s1, 0, out, N_MEL);
}

void flow_inference(cvk_ctx* ctx, const int32_t* tokens, const int* token_lens, const float* prompt_feat, const int* prompt_feat_lens,
                    const float* embedding, int B, int n_timesteps, int streaming, int finalize, float* mel, cudaStream_t st) {
  FlowModel* m = ctx->flow;
  CVK_REQUIRE(m && m->tok_emb, "flow stage not finalised");
  ctx->arena.reset();
  const int ctxl = finalize ? 0 : 3;
  // speaker embedding: F.normalize + Linear(192 -> 80) (flow.py:248-249)
  Mat en = arena_mat(ctx, DT_F32, B, 192), spk = arena_mat(ctx, DT_F32, B, N_MEL, N_MEL);
  l2norm_kernel<<<B, 64, 0, st>>>(embedding, en.f32(), 192);
  ctx->launches++;
  CVK_LAUNCH_CHECK();
  {
    Epilogue e;
    e.out = spk;
    conv_gemm_simt(ctx, st, en, m->spk_affine, e);
  }
  Seqs s2;
  Mat h = encoder_forward(ctx, st, tokens, token_lens, B, streaming, ctxl, &s2);
  Mat ha = h;
  if (ctx->act_dtype != DT_F32) {
    ha = arena_mat(ctx, ctx->act_dtype, s2.R, D_ENC);
    convert_mat(ctx, st, h, ha);
  }
  Mat mu = arena_mat(ctx, DT_F32, s2.R, N_MEL, N_MEL);
  {
    Epilogue e;
    e.row2seq = s2.d_row2seq;
    e.out = mu;
    conv_gemm(ctx, st, ha, m->enc_proj, e);
  }
  // conditions: prompt mel in the first Tp rows of every sequence, zeros elsewhere (flow.py:266-268)
  Mat cond = arena_mat(ctx, DT_F32, s2.R, N_MEL, N_MEL);
  zero_mat(ctx, st, cond);
  std::vector<int> mel_lens(B);
  for (int b = 0; b < B; ++b) {
    mel_lens[b] = s2.len[b];
    CVK_REQUIRE(prompt_feat_lens[b] >= 0 && prompt_feat_lens[b] < mel_lens[b], "prompt_feat longer than the generated mel");
  }
  if (prompt_feat) {
    Seqs sp = subseqs(ctx, s2, prompt_feat_lens, st);
    pack_rows(ctx, st, prompt_feat, N_MEL, sp, cond);
  }
  Mat x = arena_mat(ctx, DT_F32, s2.R, N_MEL, N_MEL);
  zero_mat(ctx, st, x);
  CVK_REQUIRE(m->noise && m->noise_T >= s2.max_len, "cvk_cfm_set_noise has not been called (or the noise tensor is too short)");
  {
    int bx = s2.max_len < 1024 ? s2.max_len : 1024;
    noise_init_kernel<<<dim3(bx, B), 96, 0, st>>>(m->noise, m->noise_T, s2.d_start, s2.d_len, x.f32());
    ctx->launches++;
    CVK_LAUNCH_CHECK();
  }
  cfm_solve_packed(ctx, st, s2, mel_lens.data(), mu, cond, spk.f32(), x, n_timesteps, 0.7f, streaming);
  unpack_rows_skip(ctx, st, x, s2, prompt_feat_lens, mel, N_MEL);
}

// ================================================================================================ incremental streaming flow
static Mat dit_mu_forward(cvk_ctx* ctx, cudaStream_t st, const int32_t* tokens, const int* token_lens, int B, int ctxl, Seqs* s2_out);
void flow_stream_destroy(cvk_flow_stream* fs);

// kind 0: CosyVoice2 U-Net estimator (stage "flow"); kind 1: CosyVoice3 DiT (stage "flow3").  n_slots utterances share the
// allocation; the reference gives every streaming request its own thread and recomputes its prefix (cli/model.py:343-363).
cvk_flow_stream* flow_stream_create(cvk_ctx* ctx, int kind, int n_slots, int max_frames, int n_timesteps) {
  CVK_REQUIRE(kind == 0 || kind == 1, "flow stream: unknown estimator kind");
  CVK_REQUIRE(n_slots >= 1 && max_frames >= 2 * CHUNK_TOK && n_timesteps >= 1, "flow stream: bad slot count / capacity / step count");
  cvk_flow_stream* fs = new cvk_flow_stream();
  fs->kind = kind;
  fs->cap = round_up(max_frames, 64);
  fs->n_slots = n_slots;
  fs->n_steps = n_timesteps;
  fs->adt = ctx->act_dtype;
  fs->frames_done.assign(n_slots, 0);
  fs->prompt_frames.assign(n_slots, 0);
  fs->begun.assign(n_slots, 0);
  const size_t es = fs->adt == DT_F32 ? 4 : 2;
  if (kind == 0) {
    FlowModel* m = ctx->flow;
    CVK_REQUIRE(m && m->tok_emb, "flow stage not finalised");
    const int nst = (int)m->stages.size();
    fs->n_tb = nst * m->n_blocks;
    fs->n_conv = 2 * nst + 3;
    fs->kv_width = 1024; fs->tail_rows = 2; fs->conv_c = 512;
  } else {
    DitModel* m = ctx->dit;
    CVK_REQUIRE(m && m->tok_emb, "flow3 stage not finalised");
    fs->n_tb = m->depth;
    fs->n_conv = 2;                   // the two grouped k31 position convolutions of the input embedding
    fs->kv_width = 2 * DIT_D; fs->tail_rows = DIT_CK - 1; fs->conv_c = DIT_D;
  }
  fs->kv_step_bytes = (size_t)fs->n_tb * ((size_t)2 * n_slots * fs->cap + 64) * fs->kv_width * es;
  fs->conv_step_bytes = (size_t)fs->n_conv * 2 * n_slots * fs->tail_rows * fs->conv_c * es;
  try {
    CVK_CHECK_CUDA(cudaMalloc(&fs->kv, fs->kv_step_bytes * n_timesteps));
    CVK_CHECK_CUDA(cudaMalloc(&fs->conv, fs->conv_step_bytes * n_timesteps));
    CVK_CHECK_CUDA(cudaMalloc(&fs->prompt_feat, sizeof(float) * (size_t)n_slots * fs->cap * N_MEL));
    CVK_CHECK_CUDA(cudaMalloc(&fs->spk, sizeof(float) * (size_t)n_slots * N_MEL));
    CVK_CHECK_CUDA(cudaMalloc(&fs->d_geo, sizeof(int) * 8 * n_slots));
    CVK_CHECK_CUDA(cudaMemset(fs->kv, 0, fs->kv_step_bytes * n_timesteps));   // masked key rows of a partial tile must be finite
  } catch (...) {                      // out of memory half way: give back what was taken
    cudaGetLastError();
    flow_stream_destroy(fs);
    throw;
  }
  fs->kg.d_kstart = fs->d_geo;
  fs->kg.d_klen = fs->d_geo + 2 * n_slots;
  fs->kg.d_qoff = fs->d_geo + 4 * n_slots;
  fs->d_cidx = fs->d_geo + 6 * n_slots;
  return fs;
}

void flow_stream_destroy(cvk_flow_stream* fs) {
  if (!fs) return;
  cudaFree(fs->kv); cudaFree(fs->conv); cudaFree(fs->prompt_feat); cudaFree(fs->spk); cudaFree(fs->d_geo);
  delete fs;
}

size_t flow_stream_bytes(const cvk_flow_stream* fs) { return (fs->kv_step_bytes + fs->conv_step_bytes) * (size_t)fs->n_steps; }

static void require_stage(cvk_ctx* ctx, const cvk_flow_stream* fs) {
  CVK_REQUIRE(fs->kind == 0 ? (ctx->flow && ctx->flow->tok_emb) : (ctx->dit && ctx->dit->tok_emb), "flow stage of this session not finalised");
  CVK_REQUIRE(fs->adt == ctx->act_dtype, "flow stream was created under another precision");
}

// new utterance in `slot`: prompt mel [prompt_frames][80] and speaker embedding [192] (device pointers); clears the slot's
// convolution tails (its K/V rows are overwritten chunk by chunk and never read beyond what was written)
void flow_stream_begin(cvk_ctx* ctx, cvk_flow_stream* fs, int slot, const float* prompt_feat, int prompt_frames, const float* embedding, cudaStream_t st) {
  require_stage(ctx, fs);
  const ConvW& spk_affine = fs->kind == 0 ? ctx->flow->spk_affine : ctx->dit->spk_affine;
  CVK_REQUIRE(slot >= 0 && slot < fs->n_slots, "flow stream: slot out of range");
  CVK_REQUIRE(prompt_frames >= 0 && prompt_frames < fs->cap, "flow stream: prompt longer than the cache");
  ctx->arena.reset();
  // causal left padding of the first chunk: the slot's 2 states of every (step, convolution), one pitched row each
  const size_t es = fs->adt == DT_F32 ? 4 : 2;
  const size_t state_bytes = (size_t)fs->tail_rows * fs->conv_c * es;
  CVK_CHECK_CUDA(cudaMemset2DAsync((char*)fs->conv + (size_t)2 * slot * state_bytes, (size_t)2 * fs->n_slots * state_bytes, 0, 2 * state_bytes,
                                   (size_t)fs->n_steps * fs->n_conv, st));
  if (prompt_frames > 0)
    CVK_CHECK_CUDA(cudaMemcpyAsync(fs->prompt_feat + (size_t)slot * fs->cap * N_MEL, prompt_feat, sizeof(float) * (size_t)prompt_frames * N_MEL,
                                   cudaMemcpyDeviceToDevice, st));
  Mat en = arena_mat(ctx, DT_F32, 1, 192);
  l2norm_kernel<<<1, 64, 0, st>>>(embedding, en.f32(), 192);
  ctx->launches++;
  CVK_LAUNCH_CHECK();
  {
    Epilogue e;
    e.out = Mat(fs->spk + (size_t)slot * N_MEL, DT_F32, 1, N_MEL, N_MEL);
    conv_gemm_simt(ctx, st, en, spk_affine, e);
  }
  fs->prompt_frames[slot] = prompt_frames;
  fs->frames_done[slot] = 0;
  fs->begun[slot] = 1;
}

// B begun slots advance at once.  tokens: device, B prefixes back to back (token_lens[b] each) = prompt tokens + every speech
// token so far INCLUDING the 3 look-ahead tokens (the argument the reference passes to flow.inference(streaming=True,
// finalize=False), cli/model.py:346-363).  Produces, for every slot, the mel frames that call would return beyond those already
// delivered: rows [max(frames_done, prompt_frames), 2 * (token_lens[b] - 3)), written back to back to mel_out [*, 80], their
// counts in n_out[b].  Both chunk ends must be multiples of the 50-frame static chunk (the reference's hop schedule guarantees
// it: cli/model.py:346-352 pads the first hop to the 25-token grid).  Every slot is checked before anything is launched, so a
// refused call leaves all slots as they were.
void flow_stream_chunk_batch(cvk_ctx* ctx, cvk_flow_stream* fs, int B, const int* slots, const int32_t* tokens, const int* token_lens,
                             float* mel_out, int mel_cap_frames, int* n_out, cudaStream_t st) {
  require_stage(ctx, fs);
  CVK_REQUIRE(ctx->flow && ctx->flow->noise, "cvk_cfm_set_noise has not been called");
  FlowModel* m = ctx->flow;          // holds the CFM noise for both estimator kinds
  CVK_REQUIRE(B >= 1 && B <= fs->n_slots, "flow stream: bad batch size");
  const int CH = 2 * CHUNK_TOK;
  std::vector<int> T_total(B), T_prev(B), n_new(B), skip(B), seen(fs->n_slots, 0);
  int out_frames = 0, max_total = 0;
  for (int b = 0; b < B; ++b) {
    const int sl = slots[b];
    CVK_REQUIRE(sl >= 0 && sl < fs->n_slots, "flow stream: slot out of range");
    CVK_REQUIRE(!seen[sl], "flow stream: a slot appears twice in one call");
    seen[sl] = 1;
    CVK_REQUIRE(fs->begun[sl], "cvk_flow_stream_slot_begin has not been called for this slot");
    T_total[b] = 2 * (token_lens[b] - 3);
    T_prev[b] = fs->frames_done[sl];
    CVK_REQUIRE(T_total[b] > T_prev[b], "flow stream: no new frames in this call");
    CVK_REQUIRE(T_total[b] % CH == 0 && T_prev[b] % CH == 0, "flow stream: chunk ends must be multiples of the 50-frame static chunk");
    CVK_REQUIRE(T_total[b] <= fs->cap, "flow stream: cache capacity exceeded");
    CVK_REQUIRE(fs->prompt_frames[sl] < T_total[b], "flow stream: prompt_feat longer than the generated mel");
    n_new[b] = T_total[b] - T_prev[b];
    skip[b] = fs->prompt_frames[sl] > T_prev[b] ? fs->prompt_frames[sl] - T_prev[b] : 0;   // prompt rows are computed but not returned
    out_frames += n_new[b] - skip[b];
    max_total = std::max(max_total, T_total[b]);
  }
  CVK_REQUIRE(out_frames <= mel_cap_frames, "flow stream: output buffer too small");
  CVK_REQUIRE(m->noise_T >= max_total, "the CFM noise tensor is too short");
  ctx->arena.reset();
  Seqs s2;
  Mat mu_full;
  if (fs->kind == 0) {
    // encoder over the whole prefixes (1.5 % of the flow FLOPs; its chunk mask + look-ahead make the prefix rows final as well)
    Mat h = encoder_forward(ctx, st, tokens, token_lens, B, 1, 3, &s2);
    Mat ha = h;
    if (ctx->act_dtype != DT_F32) {
      ha = arena_mat(ctx, ctx->act_dtype, s2.R, D_ENC);
      convert_mat(ctx, st, h, ha);
    }
    mu_full = arena_mat(ctx, DT_F32, s2.R, N_MEL, N_MEL);
    Epilogue e;
    e.row2seq = s2.d_row2seq;
    e.out = mu_full;
    conv_gemm(ctx, st, ha, m->enc_proj, e);
  } else {
    mu_full = dit_mu_forward(ctx, st, tokens, token_lens, B, 3, &s2);      // token embedding + look-ahead layer + x2 repeat: row-local
  }
  for (int b = 0; b < B; ++b) CVK_REQUIRE(s2.len[b] == T_total[b], "flow stream: conditioning length mismatch");
  // geometry of the new rows; per-sequence inputs gathered from each slot's position
  Seqs s1 = make_seqs(ctx, n_new.data(), B, 8, 1, 0, st);
  Mat mu = arena_mat(ctx, DT_F32, s1.R, N_MEL, N_MEL), cond = arena_mat(ctx, DT_F32, s1.R, N_MEL, N_MEL), x = arena_mat(ctx, DT_F32, s1.R, N_MEL, N_MEL);
  Mat spk = arena_mat(ctx, DT_F32, B, N_MEL, N_MEL);
  zero_mat(ctx, st, mu); zero_mat(ctx, st, cond); zero_mat(ctx, st, x);
  std::vector<int> gi(3 * B);
  for (int b = 0; b < B; ++b) {
    gi[b] = T_prev[b];
    gi[B + b] = fs->prompt_frames[slots[b]];
    gi[2 * B + b] = slots[b];
  }
  {
    const int* d_gi = upload(ctx, gi, st);
    int bx = s1.max_len < 1024 ? s1.max_len : 1024;
    stream_gather_kernel<<<dim3(bx, B), 96, 0, st>>>(mu_full.f32(), s2.d_start, m->noise, fs->prompt_feat, fs->spk, fs->cap, d_gi, B, s1.d_start,
                                                     s1.d_len, mu.f32(), cond.f32(), x.f32(), spk.f32());
    ctx->launches++;
    CVK_LAUNCH_CHECK();
  }
  // cache geometry of the 2B CFG sequences: sequence b (conditional) and b + B (unconditional) of slot s use K/V rows from
  // (2s + c) * cap and convolution state 2s + c
  const int n2 = 2 * fs->n_slots;
  std::vector<int> geo(4 * n2, 0);
  for (int b2 = 0; b2 < 2 * B; ++b2) {
    const int b = b2 % B, c = b2 / B, state = 2 * slots[b] + c;
    geo[b2] = state * fs->cap;
    geo[n2 + b2] = T_total[b];
    geo[2 * n2 + b2] = T_prev[b];
    geo[3 * n2 + b2] = state;
  }
  int* d_tmp = upload(ctx, geo, st);
  CVK_CHECK_CUDA(cudaMemcpyAsync(fs->d_geo, d_tmp, sizeof(int) * geo.size(), cudaMemcpyDeviceToDevice, st));
  cfm_solve_packed(ctx, st, s1, n_new.data(), mu, cond, spk.f32(), x, fs->n_steps, 0.7f, 1, fs->kind, fs);
  unpack_rows_skip(ctx, st, x, s1, skip.data(), mel_out, N_MEL);
  for (int b = 0; b < B; ++b) {
    fs->frames_done[slots[b]] = T_total[b];
    n_out[b] = n_new[b] - skip[b];
  }
}

// ================================================================================================ CosyVoice3 entry points
void dit_build(cvk_ctx* ctx, const int* cfg, int ncfg) {
  DitModel* m = new DitModel();
  if (ncfg >= 1) m->depth = cfg[0];
  const std::string P = "flow3.";
  m->tok_emb = copy_param(ctx, P + "input_embedding.weight");
  m->spk_affine = make_linear(ctx, P + "spk_embed_affine_layer.weight", P + "spk_embed_affine_layer.bias");
  m->spk_affine.w16 = nullptr;
  m->pre1 = make_conv_named(ctx, P + "pre_lookahead_layer.conv1.weight", P + "pre_lookahead_layer.conv1.bias", 1, 0);
  m->pre2 = make_conv_named(ctx, P + "pre_lookahead_layer.conv2.weight", P + "pre_lookahead_layer.conv2.bias", 1, -2);
  const std::string D = P + "decoder.estimator.";
  m->t1 = make_linear(ctx, D + "time_embed.time_mlp.0.weight", D + "time_embed.time_mlp.0.bias");
  m->t2 = make_linear(ctx, D + "time_embed.time_mlp.2.weight", D + "time_embed.time_mlp.2.bias");
  m->t1.w16 = nullptr;
  m->t2.w16 = nullptr;
  {
    const RawTensor& w = ctx->get_raw(D + "input_embed.proj.weight");
    CVK_REQUIRE(w.shape[0] == DIT_D && w.shape[1] == 320, "input_embed.proj must be [1024, 320]");
    float* perm = (float*)ctx->dmalloc((size_t)DIT_D * 320 * sizeof(float));
    dit_permute_inproj_kernel<<<256, 256>>>(w.p, perm, DIT_D);
    CVK_LAUNCH_CHECK();
    CVK_CHECK_CUDA(cudaDeviceSynchronize());
    m->in_proj = make_conv(ctx, perm, ctx->get_raw(D + "input_embed.proj.bias").p, DIT_D, 320, 1, 1, 0);
  }
  for (int c = 0; c < 2; ++c) {
    const std::string n = D + "input_embed.conv_pos_embed.conv" + std::to_string(c + 1) + ".0.";
    const RawTensor& w = ctx->get_raw(n + "weight");
    const RawTensor& b = ctx->get_raw(n + "bias");
    CVK_REQUIRE(w.shape[0] == DIT_D && w.shape[1] == DIT_D / DIT_GROUPS && w.shape[2] == DIT_CK, "conv_pos_embed must be [1024, 64, 31]");
    for (int g = 0; g < DIT_GROUPS; ++g) {
      ConvW cw = make_conv(ctx, w.p + (size_t)g * 64 * 64 * DIT_CK, b.p + g * 64, 64, 64, DIT_CK, 1, -(DIT_CK - 1));   // causal: 30 rows back
      (c == 0 ? m->pos1 : m->pos2).push_back(cw);
    }
  }
  std::vector<std::string> mw, mbias;
  for (int i = 0; i < m->depth; ++i) {
    const std::string b = D + "transformer_blocks." + std::to_string(i) + ".";
    mw.push_back(b + "attn_norm.linear.weight");
    mbias.push_back(b + "attn_norm.linear.bias");
    DitBlockW w;
    w.qkv = concat_linear(ctx, {b + "attn.to_q.weight", b + "attn.to_k.weight", b + "attn.to_v.weight"},
                          {b + "attn.to_q.bias", b + "attn.to_k.bias", b + "attn.to_v.bias"});
    w.out = make_linear(ctx, b + "attn.to_out.0.weight", b + "attn.to_out.0.bias");
    w.ff1 = make_linear(ctx, b + "ff.ff.0.0.weight", b + "ff.ff.0.0.bias");
    w.ff2 = make_linear(ctx, b + "ff.ff.2.weight", b + "ff.ff.2.bias");
    m->blocks.push_back(w);
  }
  mw.push_back(D + "norm_out.linear.weight");
  mbias.push_back(D + "norm_out.linear.bias");
  m->mod_all = concat_linear(ctx, mw, mbias);
  m->mod_all.w16 = nullptr;        // fp32 CUDA-core GEMM on 2B rows
  m->proj_out = make_linear(ctx, D + "proj_out.weight", D + "proj_out.bias");
  CVK_CHECK_CUDA(cudaDeviceSynchronize());
  ctx->dit = m;
}

// dit.py:145-176 on dense inputs (same argument layout as cvk_cfm_estimator)
void dit_estimator(cvk_ctx* ctx, const float* x, const float* mu, const float* t, const float* spks, const float* cond, const int* lens,
                   int B, int streaming, float* out, cudaStream_t st) {
  CVK_REQUIRE(ctx->dit && ctx->dit->tok_emb, "flow3 stage not finalised");
  ctx->arena.reset();
  const int adt = ctx->act_dtype;
  Seqs s = make_seqs(ctx, lens, B, 32, 1, 0, st);
  Mat in0 = arena_mat(ctx, adt, s.R, 320);
  zero_mat(ctx, st, in0);
  int* off = upload(ctx, prefix(lens, B), st);
  int bx = s.max_len < 1024 ? s.max_len : 1024;
  if (adt == DT_F32) est_pack_kernel<float><<<dim3(bx, B), 96, 0, st>>>(x, mu, cond, spks, off, s.d_start, s.d_len, in0.f32(), in0.ld);
  else est_pack_kernel<bf16><<<dim3(bx, B), 96, 0, st>>>(x, mu, cond, spks, off, s.d_start, s.d_len, in0.b16(), in0.ld);
  ctx->launches++;
  CVK_LAUNCH_CHECK();
  Mat v = arena_mat(ctx, DT_F32, s.R, N_MEL, N_MEL);
  dit_estimator_forward(ctx, st, s, in0, t, streaming, v, nullptr);
  unpack_rows(ctx, st, v, s, 0, out, N_MEL);
}

// flow.py:369-414 CausalMaskedDiffWithDiT.inference, batched over ragged utterances
// CosyVoice3 conditioning: token embedding (80 wide) -> PreLookaheadLayer(80, 1024, 3) -> + input -> repeat_interleave(2): mu in the
// mel geometry *s2_out (flow/flow.py:385-393, upsample_encoder.py:82-103); ctxl look-ahead tokens are consumed and dropped
static Mat dit_mu_forward(cvk_ctx* ctx, cudaStream_t st, const int32_t* tokens, const int* token_lens, int B, int ctxl, Seqs* s2_out) {
  DitModel* m = ctx->dit;
  const int adt = ctx->act_dtype;
  Seqs sf = make_seqs(ctx, token_lens, B, 8, 1, 0, st);
  Seqs s1 = ctxl > 0 ? shrink_seqs(ctx, sf, ctxl, st) : sf;
  int* toff = upload(ctx, prefix(token_lens, B), st);
  Mat emb = arena_mat(ctx, DT_F32, sf.R, N_MEL);
  zero_mat(ctx, st, emb);
  {
    int bx = sf.max_len < 512 ? sf.max_len : 512;
    token_embed_kernel<float><<<dim3(bx, B), 96, 0, st>>>(tokens, toff, m->tok_emb, sf.d_start, sf.d_len, emb.f32(), emb.ld, N_MEL);
    ctx->launches++;
    CVK_LAUNCH_CHECK();
  }
  Mat emba = emb;
  if (adt != DT_F32) {
    emba = arena_mat(ctx, adt, sf.R, N_MEL);
    convert_mat(ctx, st, emb, emba);
  }
  Mat c1 = arena_mat(ctx, adt, sf.R, DIT_D);
  {
    Epilogue e;
    e.act1 = ACT_LRELU;
    e.act1_param = 0.01f;
    e.row2seq = s1.d_row2seq;
    e.out = c1;
    conv_gemm(ctx, st, emba, m->pre1, e);
  }
  Mat h = arena_mat(ctx, DT_F32, sf.R, N_MEL);
  {
    Epilogue e;
    e.resid = emb;
    e.row2seq = s1.d_row2seq;      // look-ahead context rows are dropped here
    e.out = h;
    conv_gemm(ctx, st, c1, m->pre2, e);
  }
  // mu = repeat_interleave(h, 2) in the mel geometry
  Seqs s2 = scale_seqs(ctx, s1, 2, 0, st);
  Mat mu = arena_mat(ctx, DT_F32, s2.R, N_MEL, N_MEL);
  zero_mat(ctx, st, mu);
  {
    int bx = s1.max_len < 1024 ? s1.max_len : 1024;
    repeat2_rows_kernel<<<dim3(bx, B), 96, 0, st>>>(h.f32(), h.ld, s1.d_start, s1.d_len, mu.f32(), mu.ld, s2.d_start, N_MEL);
    ctx->launches++;
    CVK_LAUNCH_CHECK();
  }
  *s2_out = s2;
  return mu;
}

void flow3_inference(cvk_ctx* ctx, const int32_t* tokens, const int* token_lens, const float* prompt_feat, const int* prompt_feat_lens,
                     const float* embedding, int B, int n_timesteps, int streaming, int finalize, float* mel, cudaStream_t st) {
  DitModel* m = ctx->dit;
  CVK_REQUIRE(m && m->tok_emb, "flow3 stage not finalised");
  CVK_REQUIRE(ctx->flow && ctx->flow->noise, "cvk_cfm_set_noise has not been called");
  ctx->arena.reset();
  const int adt = ctx->act_dtype;
  const int ctxl = finalize ? 0 : 3;
  Mat en = arena_mat(ctx, DT_F32, B, 192), spk = arena_mat(ctx, DT_F32, B, N_MEL, N_MEL);
  l2norm_kernel<<<B, 64, 0, st>>>(embedding, en.f32(), 192);
  ctx->launches++;
  CVK_LAUNCH_CHECK();
  {
    Epilogue e;
    e.out = spk;
    conv_gemm_simt(ctx, st, en, m->spk_affine, e);
  }
  Seqs s2;
  Mat mu = dit_mu_forward(ctx, st, tokens, token_lens, B, ctxl, &s2);
  Mat cond = arena_mat(ctx, DT_F32, s2.R, N_MEL, N_MEL);
  zero_mat(ctx, st, cond);
  std::vector<int> mel_lens(B);
  for (int b = 0; b < B; ++b) {
    mel_lens[b] = s2.len[b];
    CVK_REQUIRE(prompt_feat_lens[b] >= 0 && prompt_feat_lens[b] < mel_lens[b], "prompt_feat longer than the generated mel");
  }
  if (prompt_feat) {
    Seqs sp = subseqs(ctx, s2, prompt_feat_lens, st);
    pack_rows(ctx, st, prompt_feat, N_MEL, sp, cond);
  }
  Mat x = arena_mat(ctx, DT_F32, s2.R, N_MEL, N_MEL);
  zero_mat(ctx, st, x);
  CVK_REQUIRE(ctx->flow->noise_T >= s2.max_len, "the CFM noise tensor is too short");
  {
    int bx = s2.max_len < 1024 ? s2.max_len : 1024;
    noise_init_kernel<<<dim3(bx, B), 96, 0, st>>>(ctx->flow->noise, ctx->flow->noise_T, s2.d_start, s2.d_len, x.f32());
    ctx->launches++;
    CVK_LAUNCH_CHECK();
  }
  cfm_solve_packed(ctx, st, s2, mel_lens.data(), mu, cond, spk.f32(), x, n_timesteps, 0.7f, streaming, 1);
  unpack_rows_skip(ctx, st, x, s2, prompt_feat_lens, mel, N_MEL);
}
