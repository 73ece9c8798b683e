// Internal definitions shared by the libcvk translation units (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>
#include <map>
#include <unordered_map>
#include <stdexcept>
#include <atomic>

#include "../../include/cvk.h"

typedef __nv_bfloat16 bf16;

// ------------------------------------------------------------------------------------------------ errors
struct CvkError : std::runtime_error {
  int code;
  CvkError(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

#define CVK_CHECK_CUDA(expr)                                                                       \
  do {                                                                                             \
    cudaError_t _e = (expr);                                                                       \
    if (_e != cudaSuccess)                                                                         \
      throw CvkError(CVK_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e) + " @" +     \
                                       __FILE__ + ":" + std::to_string(__LINE__));                 \
  } while (0)

#define CVK_REQUIRE(cond, msg)                                                                     \
  do {                                                                                             \
    if (!(cond))                                                                                   \
      throw CvkError(CVK_ERR_INVALID, std::string(msg) + " (" #cond ") @" + __FILE__ + ":" +       \
                                          std::to_string(__LINE__));                               \
  } while (0)

#define CVK_LAUNCH_CHECK() CVK_CHECK_CUDA(cudaGetLastError())

// ------------------------------------------------------------------------------------------------ tensors
// DT_F16: IEEE half operands (10-bit mantissa) - used for the vocoder stage in the tensor-core mode: the reference keeps HiFT in
// "fp32", i.e. on the GPU cuDNN's default TF32 convolutions (10-bit mantissa as well); bf16 (7 bits) would be narrower than that.
enum DType { DT_F32 = 0, DT_BF16 = 1, DT_F16 = 2 };

// A 2-D row-major view [rows, cols] with row pitch ld (elements).  Activations are time-major: one row per
// frame / token / sample-block, channels contiguous.
struct Mat {
  void* p = nullptr;
  int dtype = DT_F32;
  int rows = 0;
  int cols = 0;
  int ld = 0;
  Mat() {}
  Mat(void* p_, int dt, int r, int c, int ld_) : p(p_), dtype(dt), rows(r), cols(c), ld(ld_) {}
  size_t esize() const { return dtype == DT_F32 ? 4 : 2; }
  // column slice [c0, c0+n)
  Mat slice(int c0, int n) const { return Mat((char*)p + (size_t)c0 * esize(), dtype, rows, n, ld); }
  float* f32() const { return (float*)p; }
  bf16* b16() const { return (bf16*)p; }
};

// Packed ragged batch geometry.  Sequence b occupies rows [start[b], start[b]+len[b]) of every activation
// matrix at this rate; all other rows ("gap rows") hold zeros so that convolution halos read zeros
// (the reference multiplies by the padding mask after every block, flow/decoder.py:65-78).
struct Seqs {
  int B = 0;
  int R = 0;                      // total rows (multiple of 128)
  std::vector<int> start, len;    // host copies
  int* d_start = nullptr;         // [B]
  int* d_len = nullptr;           // [B]
  int* d_row2seq = nullptr;       // [R]  sequence index or -1 for gap rows
  int max_len = 0;
  int64_t sum_len = 0;
};

// Weight of a (dilated / causal / transposed-as-polyphase) 1-D convolution or a Linear layer, repacked to
// [N][taps][K] (K contiguous).  out[r, n] = bias[n] + sum_j sum_k A[r + shift0 + j*dil, k] * w[n][j][k]
struct ConvW {
  int N = 0, K = 0, taps = 1, dil = 1, shift0 = 0;
  float* w32 = nullptr;   // always present
  bf16* w16 = nullptr;    // present in bf16 mode
  __half* wf16 = nullptr; // IEEE-half copy instead of w16 (vocoder weights when the stage runs on fp16 operands)
  float* bias = nullptr;  // [N] or null
};

enum Act {
  ACT_NONE = 0, ACT_GELU = 1, ACT_SILU = 2, ACT_MISH = 3, ACT_ELU = 4, ACT_LRELU = 5, ACT_SNAKE = 6, ACT_TANH = 7, ACT_ABS = 8,
  ACT_GELU_TANH = 9   // F.gelu(approximate='tanh') (CosyVoice3 DiT feed-forward, flow/DiT/modules.py:514)
};

// Fused epilogue of the conv-GEMM kernels:
//   v = acc + bias[n] + rowvec[seq(r)][n]            (rowvec: per-sequence broadcast add, e.g. time-MLP)
//   v = act1(v) * scale
//   v = v + resid[r][n]
//   v = valid(r) ? v : 0
//   out  = accumulate ? out + v : v                   (fp32 or bf16)
//   out2 = valid(r) ? act2(v) : 0                     (optional second output, e.g. next Snake-activated operand)
struct Epilogue {
  const float* bias = nullptr;
  const float* rowvec = nullptr;  // [B][rowvec_ld]
  int rowvec_ld = 0;
  int act1 = ACT_NONE;
  float act1_param = 0.f;          // lrelu slope
  const float* alpha1 = nullptr;   // snake alpha per column
  float scale = 1.f;
  Mat resid;                       // fp32, optional
  const int* row2seq = nullptr;    // validity mask (null = all rows valid)
  int accumulate = 0;
  Mat out;                         // required
  int act2 = ACT_NONE;
  float act2_param = 0.f;
  const float* alpha2 = nullptr;
  Mat out2;                        // optional
};

// ------------------------------------------------------------------------------------------------ context
// set while the calling thread captures the LM decode step into a CUDA graph (per thread: an LM session call and a workspace
// call - flow / vocoder - may run concurrently on two host threads, see include/cvk.h)
extern thread_local int cvk_in_capture;

struct Arena {
  char* base = nullptr;
  size_t cap = 0, off = 0, high = 0;
  void* alloc(size_t bytes) {
    size_t a = (off + 255) & ~(size_t)255;
    if (a + bytes > cap) throw CvkError(CVK_ERR_OOM, "workspace arena exhausted: need " + std::to_string(a + bytes) +
                                                          " of " + std::to_string(cap));
    off = a + bytes;
    if (off > high) high = off;
    return base + a;
  }
  void reset() { off = 0; }
};

struct RawTensor {
  float* p = nullptr;  // device fp32
  std::vector<int64_t> shape;
  int64_t numel() const { int64_t n = 1; for (auto s : shape) n *= s; return n; }
};

// optional per-kernel-family timing (bench.py roofline): CUDA events around every launch of a family
enum ProfFamily { FAM_GEMM_TC = 0, FAM_GEMM_SIMT = 1, FAM_ATTN = 2, FAM_COUNT = 3 };
struct ProfRec {
  cudaEvent_t a, b;
  int family;
  double work;    // algorithmic FLOPs of the launch
  double bytes;   // algorithmic bytes of the launch
};

struct HiftModel;
struct FlowModel;
struct DitModel;
struct LlmModel;

struct cvk_ctx {
  int device = 0;
  int precision = CVK_PREC_FP32;
  int act_dtype = DT_F32;
  int num_sms = 148;
  std::string last_error;
  std::map<std::string, RawTensor> raw;     // tensors handed over by cvk_set_tensor, consumed by cvk_finalize
  std::vector<void*> owned;                 // device allocations owned by the context
  Arena arena;
  HiftModel* hift = nullptr;
  HiftModel* hift3 = nullptr;               // CosyVoice3 causal vocoder (stage "hift3"), same conv-GEMM body with causal weights
  void* hift3_extra = nullptr;              // fp64 f0 predictor + stored source noise (hift.cu)
  FlowModel* flow = nullptr;
  DitModel* dit = nullptr;                  // CosyVoice3 flow (stage "flow3")
  LlmModel* llm = nullptr;
  void* mel_model = nullptr;
  void* prompt_feat_model = nullptr;      // prompt_feat.cu (whisper log-mel / kaldi fbank constants), built on first use
  void* encode_tiled = nullptr;             // cuTensorMapEncodeTiled entry point
  std::atomic<int64_t> launches{0};         // kernels launched by this library (bench.py gpu_launches); LM-session calls and workspace calls may run on two threads
  int op_out_bf16 = 0;                      // cvk_op_conv1d: bf16 output matrix (the estimator's usual epilogue) instead of fp32
  int op_iters = 0;                         // cvk_op_conv1d: repeat the GEMM launch this many times and time it
  double op_ms = 0.0;
  int tc_epi = 2;                           // tcgen05 GEMM epilogue: 2 = smem-staged TMA stores, 0 = direct stores, 1 = direct + prefetch
  int tc_persist = 2;                       // tcgen05 GEMM, tiles > SMs: persistent CTAs + double-buffered TMEM accumulators (2 = 16 epilogue warps, 1 = 8, 0 = off)
  int tc_pbn256 = 1;                        // persistent tcgen05 GEMM: 128x256 tiles for 16-bit outputs with N % 256 == 0 (halves the A re-reads out of L2)
  int tc_bn256 = 0;                         // experiment: 128x256 tiles (1 CTA/SM) instead of 128x128 (2 CTAs/SM)
  void* dbg = nullptr;                      // device int64[1024] timeline buffer (debug option)
  void* tl = nullptr;                       // device int64[4096] LM-chain timeline (debug option chain_timeline): 4 slots per launch
  int tl_seq = 0;
  long long* tl_next() {                    // slot block of the next launch of the decode chain (null when the option is off)
    if (!tl) return nullptr;
    long long* p = (long long*)tl + 4 * (tl_seq % 1024);
    ++tl_seq;
    return p;
  }
  int prof_on = 0;
  std::vector<ProfRec> prof;
  std::unordered_map<const void*, void*> tiled;   // bf16 weight -> streaming (pre-tiled, pre-swizzled) copy for the skinny GEMM
  std::vector<cudaEvent_t> event_pool;
  int pdl = 1;                              // LM decode chain: programmatic dependent launch (next kernel's prologue + weight prefetch overlap this kernel)
  int lm_fused = 1;                         // LM decode: fused finish+rmsnorm / rope+attention / SwiGLU-epilogue kernels
  int hift_f16 = 1;                         // tensor-core mode: vocoder operands in IEEE half (TF32-class mantissa) instead of bf16
  int build_f16 = 0;                        // set while a stage whose weights need the half copy is being finalised
  int enc_tc_attn = 1;                      // conformer relative-position attention on the tcgen05 kernels (attention_tc.cu) instead of CUDA cores
  int attn_single_pass = 1;                 // flow attention: one-pass kernel with per-thread lazy maxima (attention_tc.cu)
  int lm_mega = 0;                          // LM decode: all layers of a step in one persistent cooperative kernel (llm_mega.cu); measured
                                            // 973 us / step against 886 us for the PDL-chained per-op path at batch 32 (profiles/r02_lm_decode.md): off by default
  int mega_coop = 1;                        // ... launched with the cooperative attribute (co-residency guaranteed by the driver)
  int use_skinny = 1;                       // LM decode GEMMs on the weight-streaming split-K kernel
  int use_tc_attn = 1;                      // bf16 mode: tcgen05 attention kernel (0 = CUDA-core flash kernel)
  int use_graph = 1;                        // LM decode step replayed as a CUDA graph
  int use_tc = 1;                           // bf16 mode: route GEMMs to the tcgen05 kernel (0 = debug: SIMT on converted operands)

  void* dmalloc(size_t bytes) {
    void* p = nullptr;
    CVK_CHECK_CUDA(cudaMalloc(&p, bytes ? bytes : 16));
    owned.push_back(p);
    return p;
  }
  const RawTensor& get_raw(const std::string& name) const {
    auto it = raw.find(name);
    if (it == raw.end()) throw CvkError(CVK_ERR_MISSING_WEIGHT, "missing weight tensor: " + name);
    return it->second;
  }
  bool has_raw(const std::string& name) const { return raw.find(name) != raw.end(); }
};

// kernel launch with the optional PDL attribute (see common.cuh pdl_wait/pdl_trigger)
template <typename... KArgs, typename... Args>
inline void launch_ex(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  if (pdl) {
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
  }
  CVK_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, KArgs(std::forward<Args>(args))...));
}

// ------------------------------------------------------------------------------------------------ shared ops
// geometry
Seqs make_seqs(cvk_ctx* ctx, const int* lens, int B, int gap, int scale, int extra_front, cudaStream_t st, bool with_row2seq = true);
Seqs scale_seqs(cvk_ctx* ctx, const Seqs& s, int scale, int extra_front, cudaStream_t st, bool with_row2seq = true);

// weights
ConvW make_linear(cvk_ctx* ctx, const std::string& wname, const std::string& bname);
ConvW make_conv(cvk_ctx* ctx, const float* w_oik /*[N][K][taps] device*/, const float* bias, int N, int K, int taps,
                int dil, int shift0);
ConvW make_conv_named(cvk_ctx* ctx, const std::string& wname, const std::string& bname, int dil, int shift0);
float* fold_weight_norm(cvk_ctx* ctx, const std::string& prefix, int64_t* numel_out);
void finish_convw(cvk_ctx* ctx, ConvW& w);   // create bf16 copy if needed
float* dev_copy_f32(cvk_ctx* ctx, const float* src_dev, size_t n);

// conv-GEMM (dispatches SIMT fp32 / tcgen05 bf16 on A.dtype)
void conv_gemm(cvk_ctx* ctx, cudaStream_t st, const Mat& A, const ConvW& W, const Epilogue& ep);
void conv_gemm_simt(cvk_ctx* ctx, cudaStream_t st, const Mat& A, const ConvW& W, const Epilogue& ep);
void conv_gemm_tc(cvk_ctx* ctx, cudaStream_t st, const Mat& A, const ConvW& W, const Epilogue& ep);
size_t skinny_scratch_floats(int rows, int maxN);
const bf16* skinny_tiled_weights(cvk_ctx* ctx, const ConvW& W);
void skinny_set_carveout();
int conv_gemm_skinny_ex(cvk_ctx* ctx, cudaStream_t st, const Mat& A, const ConvW& W, const Epilogue& ep, float* scratch, size_t scratch_floats,
                        int mode);
void conv_gemm_skinny(cvk_ctx* ctx, cudaStream_t st, const Mat& A, const ConvW& W, const Epilogue& ep, float* scratch, size_t scratch_floats);

// elementwise / normalisation (elementwise.cu)
void zero_mat(cvk_ctx* ctx, cudaStream_t st, const Mat& m);
// out = valid(r) ? act(LN(x)) * post_scale + rowvec[seq(r)] : 0
void layernorm(cvk_ctx* ctx, cudaStream_t st, const Mat& x, const float* gamma, const float* beta, float eps, int act,
               float post_scale, const int* row2seq, const Mat& out, const float* rowvec = nullptr, int rowvec_ld = 0);
void unpack_rows_skip(cvk_ctx* ctx, cudaStream_t st, const Mat& in, const Seqs& s, const int* skip_host, float* dense, int C);
Seqs shrink_seqs(cvk_ctx* ctx, const Seqs& s, int drop_tail, cudaStream_t st);
Seqs subseqs(cvk_ctx* ctx, const Seqs& s, const int* skip_host, cudaStream_t st);
void rmsnorm(cvk_ctx* ctx, cudaStream_t st, const Mat& x, const float* gamma, float eps, const Mat& out);
void act_copy(cvk_ctx* ctx, cudaStream_t st, const Mat& x, int act, float param, const float* alpha, const int* row2seq,
              const Mat& out);
void act_copy_scaled(cvk_ctx* ctx, cudaStream_t st, const Mat& x, float pre_scale, int act, float param, const float* alpha,
                     const int* row2seq, const Mat& out);
void pack_rows(cvk_ctx* ctx, cudaStream_t st, const float* dense, int C, const Seqs& s, const Mat& out);
void unpack_rows(cvk_ctx* ctx, cudaStream_t st, const Mat& in, const Seqs& s, int skip, float* dense, int C);
void bcast_rows(cvk_ctx* ctx, cudaStream_t st, const float* vec, int C, int vec_ld, const Seqs& s, const Mat& out);
void convert_mat(cvk_ctx* ctx, cudaStream_t st, const Mat& in, const Mat& out);

// attention (attention.cu)
//  q,k,v: packed [R, H*64] views (same Seqs); mask: key j visible from query i iff j < klimit(i), with
//  klimit(i) = len (chunk<=0) or min(len, (i/chunk+1)*chunk) (block-causal, utils/mask.py:155-157)
// Keys / values living in a cache with their own row geometry (incremental streaming flow): sequence b's keys are rows
// [kstart[b], kstart[b] + klen[b]) of the k / v matrices and its queries (rows of `s`) sit at absolute positions qoff[b] + i.
struct KvGeom {
  const int* d_kstart = nullptr;
  const int* d_klen = nullptr;
  const int* d_qoff = nullptr;
};
// prompt-side acoustic features (prompt_feat.cu)
void whisper_log_mel(cvk_ctx* ctx, const float* wav, const int* lens, int B, float* out, cudaStream_t st);
void kaldi_fbank80(cvk_ctx* ctx, const float* wav, const int* lens, int B, int subtract_mean, float* out, cudaStream_t st);
// incremental streaming flow (flow.cu)
struct cvk_flow_stream;
cvk_flow_stream* flow_stream_create(cvk_ctx* ctx, int kind, int n_slots, int max_frames, int n_timesteps);
void flow_stream_destroy(cvk_flow_stream* fs);
size_t flow_stream_bytes(const cvk_flow_stream* fs);
void flow_stream_begin(cvk_ctx* ctx, cvk_flow_stream* fs, int slot, const float* prompt_feat, int prompt_frames, const float* embedding,
                       cudaStream_t st);
void flow_stream_chunk_batch(cvk_ctx* ctx, cvk_flow_stream* fs, int B, const int* slots, const int32_t* tokens, const int* token_lens,
                             float* mel_out, int mel_cap_frames, int* n_out, cudaStream_t st);
void attention_fwd(cvk_ctx* ctx, cudaStream_t st, const Mat& q, const Mat& k, const Mat& v, const Seqs& s, int H, int chunk,
                   float scale, const Mat& out, int kv_div = 1, const KvGeom* kg = nullptr);
void relpos_attention_fwd(cvk_ctx* ctx, cudaStream_t st, const Mat& q, const Mat& k, const Mat& v, const Mat& pos /*[2*Tmax-1, H*64]*/,
                          int pos_center, const float* bias_u, const float* bias_v, const Seqs& s, int H, int chunk, float scale,
                          const Mat& out);

struct ProfScope {
  cvk_ctx* ctx;
  cudaStream_t st;
  ProfRec rec;
  bool on;
  ProfScope(cvk_ctx* c, cudaStream_t s, int family, double work, double bytes) : ctx(c), st(s), on(c->prof_on && !cvk_in_capture) {
    if (!on) return;
    auto get = [&]() {
      cudaEvent_t e;
      if (!ctx->event_pool.empty()) { e = ctx->event_pool.back(); ctx->event_pool.pop_back(); }
      else cudaEventCreate(&e);
      return e;
    };
    rec.a = get(); rec.b = get(); rec.family = family; rec.work = work; rec.bytes = bytes;
    cudaEventRecord(rec.a, st);
  }
  ~ProfScope() {
    if (!on) return;
    cudaEventRecord(rec.b, st);
    ctx->prof.push_back(rec);
  }
};

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
static inline int round_up(int a, int b) { return ceil_div(a, b) * b; }

inline Mat arena_mat(cvk_ctx* ctx, int dtype, int rows, int cols, int ld = 0) {
  if (ld == 0) ld = round_up(cols, 8);
  size_t es = dtype == DT_F32 ? 4 : 2;
  void* p = ctx->arena.alloc((size_t)rows * ld * es);
  return Mat(p, dtype, rows, cols, ld);
}
