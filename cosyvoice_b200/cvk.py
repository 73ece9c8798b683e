"""ctypes binding of libcvk.so (include/cvk.h).  PyTorch is used only as the allocator / stream provider:
tensors are passed as raw device pointers + explicit shapes, nothing here computes.

There is no CPU or eager fallback: if the shared library or a CUDA device is missing every entry point raises.
"""
import ctypes
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "lib", "libcvk.so")

PREC_FP32, PREC_BF16 = 0, 1
ACT = dict(none=0, gelu=1, silu=2, mish=3, elu=4, lrelu=5, snake=6, tanh=7, abs=8)

_lib = None
_lib_lock = threading.Lock()

_c_int_p = ctypes.POINTER(ctypes.c_int)
_vp = ctypes.c_void_p

# name -> (restype, argtypes); mirrors include/cvk.h one to one (tests/test_abi.py checks every symbol resolves)
SIGNATURES = {
    "cvk_create": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_size_t, ctypes.POINTER(_vp)]),
    "cvk_destroy": (None, [_vp]),
    "cvk_last_error": (ctypes.c_char_p, [_vp]),
    "cvk_version": (ctypes.c_char_p, []),
    "cvk_launch_count": (ctypes.c_int64, [_vp]),
    "cvk_last_op_ms": (ctypes.c_double, [_vp]),
    "cvk_debug_read": (ctypes.c_int, [_vp, ctypes.POINTER(ctypes.c_longlong), ctypes.c_int]),
    "cvk_set_option": (ctypes.c_int, [_vp, ctypes.c_char_p, ctypes.c_int]),
    "cvk_profile": (ctypes.c_int, [_vp, ctypes.c_int]),
    "cvk_profile_read": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double),
                                        ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int64)]),
    "cvk_set_tensor": (ctypes.c_int, [_vp, ctypes.c_char_p, _vp, ctypes.c_int, ctypes.POINTER(ctypes.c_int64), ctypes.c_int]),
    "cvk_finalize": (ctypes.c_int, [_vp, ctypes.c_char_p, _c_int_p, ctypes.c_int]),
    "cvk_op_conv1d": (ctypes.c_int, [_vp, _vp, _c_int_p, ctypes.c_int, ctypes.c_int, _vp, _vp, ctypes.c_int, ctypes.c_int,
                                     ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp, _vp]),
    "cvk_op_linear_small": (ctypes.c_int, [_vp, _vp, ctypes.c_int, ctypes.c_int, _vp, _vp, ctypes.c_int, _vp, ctypes.c_int,
                                           ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_longlong), _vp]),
    "cvk_op_attention": (ctypes.c_int, [_vp, _vp, _vp, _vp, _c_int_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float, _vp, _vp]),
    "cvk_hift_f0": (ctypes.c_int, [_vp, _vp, _c_int_p, ctypes.c_int, _vp, _vp]),
    "cvk_hift_source": (ctypes.c_int, [_vp, _vp, _c_int_p, ctypes.c_int, _vp, _vp, _vp]),
    "cvk_hift_decode": (ctypes.c_int, [_vp, _vp, _c_int_p, ctypes.c_int, _vp, _vp, _vp]),
    "cvk_hift_inference": (ctypes.c_int, [_vp, _vp, _c_int_p, ctypes.c_int, _vp, _vp, _c_int_p, _vp, _vp, _vp]),
    "cvk_flow_encoder": (ctypes.c_int, [_vp, _vp, _c_int_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp, _vp]),
    "cvk_cfm_estimator": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _c_int_p, ctypes.c_int, ctypes.c_int, _vp, _vp]),
    "cvk_cfm_estimator_inplace": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _c_int_p, ctypes.c_int, ctypes.c_int, _vp]),
    "cvk_workspace_bytes": (ctypes.c_int, [_vp, ctypes.POINTER(ctypes.c_size_t), ctypes.POINTER(ctypes.c_size_t)]),
    "cvk_cfm_solve": (ctypes.c_int, [_vp, _vp, _vp, _vp, _c_int_p, ctypes.c_int, _vp, ctypes.c_int, ctypes.c_float, ctypes.c_int, _vp, _vp]),
    "cvk_flow_inference": (ctypes.c_int, [_vp, _vp, _c_int_p, _vp, _c_int_p, _vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp, _vp]),
    "cvk_flow_stream_create": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, ctypes.POINTER(_vp)]),
    "cvk_flow3_stream_create": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, ctypes.POINTER(_vp)]),
    "cvk_flow_stream_destroy": (None, [_vp, _vp]),
    "cvk_flow_stream_bytes": (ctypes.c_longlong, [_vp]),
    "cvk_flow_stream_begin": (ctypes.c_int, [_vp, _vp, _vp, ctypes.c_int, _vp, _vp]),
    "cvk_flow_stream_chunk": (ctypes.c_int, [_vp, _vp, _vp, ctypes.c_int, _vp, ctypes.c_int, _c_int_p, _vp]),
    "cvk_flow_stream_slots_create": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(_vp)]),
    "cvk_flow_stream_slot_begin": (ctypes.c_int, [_vp, _vp, ctypes.c_int, _vp, ctypes.c_int, _vp, _vp]),
    "cvk_flow_stream_chunk_batch": (ctypes.c_int, [_vp, _vp, ctypes.c_int, _c_int_p, _vp, _c_int_p, _vp, ctypes.c_int, _c_int_p, _vp]),
    "cvk_cfm_set_noise": (ctypes.c_int, [_vp, _vp, ctypes.c_int, ctypes.c_int]),
    "cvk_hift3_set_noise": (ctypes.c_int, [_vp, _vp, _vp, ctypes.c_longlong, ctypes.c_int]),
    "cvk_hift3_inference": (ctypes.c_int, [_vp, _vp, _c_int_p, ctypes.c_int, ctypes.c_int, _vp, _vp, _vp, _vp]),
    "cvk_dit_estimator": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _c_int_p, ctypes.c_int, ctypes.c_int, _vp, _vp]),
    "cvk_flow3_inference": (ctypes.c_int, [_vp, _vp, _c_int_p, _vp, _c_int_p, _vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp, _vp]),
    "cvk_lm_session_create": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, ctypes.POINTER(_vp)]),
    "cvk_lm_session_destroy": (None, [_vp, _vp]),
    "cvk_lm_prefill": (ctypes.c_int, [_vp, _vp, _vp, _c_int_p, _vp, _c_int_p, ctypes.c_int, _vp]),
    "cvk_lm_decode": (ctypes.c_int, [_vp, _vp, ctypes.c_int, _vp, _vp, _vp, _vp, ctypes.c_int, _vp, _vp, _c_int_p, _vp]),
    "cvk_lm_forward_logp": (ctypes.c_int, [_vp, _vp, _c_int_p, ctypes.c_int, _vp, _vp]),
    "cvk_lm_last_logits": (ctypes.c_int, [_vp, _vp, _vp, _vp]),
    "cvk_lm_vocab": (ctypes.c_int, [_vp]),
    "cvk_lm_begin": (ctypes.c_int, [_vp, _vp, ctypes.c_int, _vp]),
    "cvk_lm_feed": (ctypes.c_int, [_vp, _vp, _c_int_p, _c_int_p, ctypes.c_int, _vp]),
    "cvk_lm_next_logp": (ctypes.c_int, [_vp, _vp, _vp, _vp]),
    "cvk_ras_sample": (ctypes.c_int, [_vp, _vp, ctypes.c_int, ctypes.c_int, _vp, ctypes.c_int, _vp, _vp, _vp, _vp, _vp]),
    "cvk_mel_spectrogram": (ctypes.c_int, [_vp, _vp, _c_int_p, ctypes.c_int, _vp, _vp]),
    "cvk_mel_spectrogram_ex": (ctypes.c_int, [_vp, _vp, _c_int_p, ctypes.c_int, ctypes.c_int, _vp, _vp]),
    "cvk_whisper_log_mel": (ctypes.c_int, [_vp, _vp, _c_int_p, ctypes.c_int, _vp, _vp]),
    "cvk_kaldi_fbank": (ctypes.c_int, [_vp, _vp, _c_int_p, ctypes.c_int, ctypes.c_int, _vp, _vp]),
}


def lib_path():
    return _LIB_PATH


def load_library():
    """dlopen libcvk.so and bind every symbol of include/cvk.h.  Raises if the library has not been built."""
    global _lib
    with _lib_lock:
        if _lib is None:
            if not os.path.exists(_LIB_PATH):
                raise RuntimeError(f"{_LIB_PATH} not found - run `python -m cosyvoice_b200.build` (needs nvcc); "
                                   "there is no CPU fallback")
            lib = ctypes.CDLL(_LIB_PATH)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(lib, name)
                fn.restype = res
                fn.argtypes = args
            _lib = lib
    return _lib


def _ints(v):
    v = [int(x) for x in v]
    return (ctypes.c_int * len(v))(*v)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _f32(t, device):
    return t.to(device=device, dtype=torch.float32).contiguous()


class CvkError(RuntimeError):
    pass


class Context:
    """One cvk_ctx per (process, GPU)."""

    def __init__(self, device=0, precision="bf16", workspace_gb=4.0):
        if not torch.cuda.is_available():
            raise RuntimeError("cosyvoice_b200 requires a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = load_library()
        self.device = torch.device("cuda", device)
        self.precision = PREC_BF16 if precision in ("bf16", PREC_BF16) else PREC_FP32
        h = ctypes.c_void_p()
        torch.cuda.set_device(self.device)
        torch.zeros(1, device=self.device)           # make sure the primary context exists
        rc = self.lib.cvk_create(device, self.precision, int(workspace_gb * (1 << 30)), ctypes.byref(h))
        if rc != 0:
            raise CvkError(f"cvk_create failed with status {rc} (needs an sm_100 GPU)")
        self.h = h
        self.lock = threading.Lock()

    def close(self):
        if getattr(self, "h", None):
            self.lib.cvk_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            msg = self.lib.cvk_last_error(self.h)
            raise CvkError(f"libcvk status {rc}: {msg.decode() if msg else ''}")

    # ------------------------------------------------------------------ weights
    def load_state_dict(self, stage, state_dict, cfg=()):
        """Hand a reference state_dict (fp32) to the library and finalise the stage."""
        torch.cuda.synchronize(self.device)
        for k, v in state_dict.items():
            if not torch.is_tensor(v) or not v.dtype.is_floating_point:
                continue
            if stage == "llm" and k == "llm.model.lm_head.weight":
                continue      # tied alias of embed_tokens, never used at inference (llm/llm.py:542 uses llm_decoder)
            t = v.detach().to(dtype=torch.float32).contiguous()
            on_dev = 1 if t.is_cuda else 0
            shape = (ctypes.c_int64 * max(t.dim(), 1))(*(list(t.shape) or [1]))
            self._check(self.lib.cvk_set_tensor(self.h, f"{stage}.{k}".encode(), _ptr(t), on_dev, shape, max(t.dim(), 1)))
        self.finalize(stage, cfg)

    def finalize(self, stage, cfg=()):
        cfg = list(cfg)
        self._check(self.lib.cvk_finalize(self.h, stage.encode(), _ints(cfg) if cfg else None, len(cfg)))

    def set_option(self, key, value):
        self._check(self.lib.cvk_set_option(self.h, key.encode(), int(value)))

    def profile(self, enable):
        self._check(self.lib.cvk_profile(self.h, int(enable)))

    def profile_read(self, family):
        ms, fl, by, n = ctypes.c_double(), ctypes.c_double(), ctypes.c_double(), ctypes.c_int64()
        self._check(self.lib.cvk_profile_read(self.h, family, ctypes.byref(ms), ctypes.byref(fl), ctypes.byref(by), ctypes.byref(n)))
        return dict(ms=ms.value, flops=fl.value, bytes=by.value, launches=n.value)

    def debug_read(self, n=1024):
        buf = (ctypes.c_longlong * n)()
        self._check(self.lib.cvk_debug_read(self.h, buf, n))
        return list(buf)

    def last_op_ms(self):
        return float(self.lib.cvk_last_op_ms(self.h))

    def launch_count(self):
        return int(self.lib.cvk_launch_count(self.h))

    # ------------------------------------------------------------------ generic ops (tests)
    def conv1d(self, x, lens, w, bias, dil=1, shift0=0, act="none"):
        """x [sum(lens), K] time-major; w torch Conv1d weight [N,K,taps]."""
        x = _f32(x, self.device)
        w = _f32(w, self.device)
        b = _f32(bias, self.device) if bias is not None else None
        N, K, taps = w.shape
        out = torch.empty(x.shape[0], N, device=self.device)
        self._check(self.lib.cvk_op_conv1d(self.h, _ptr(x), _ints(lens), len(lens), K, _ptr(w), _ptr(b), N, taps, dil, shift0,
                                           ACT[act], _ptr(out), _stream()))
        return out

    def linear_small(self, x, w, bias=None, iters=0, timeline=False):
        x, w = _f32(x, self.device), _f32(w, self.device)
        b = _f32(bias, self.device) if bias is not None else None
        out = torch.empty(x.shape[0], w.shape[0], device=self.device)
        ms = ctypes.c_float(0)
        tl = (ctypes.c_longlong * 1024)() if timeline else None
        self._check(self.lib.cvk_op_linear_small(self.h, _ptr(x), x.shape[0], x.shape[1], _ptr(w), _ptr(b), w.shape[0], _ptr(out), iters,
                                                 ctypes.byref(ms), tl, _stream()))
        return out, ms.value, (list(tl) if timeline else None)

    def attention(self, q, k, v, lens, heads, chunk=0, scale=0.125):
        q, k, v = (_f32(t, self.device) for t in (q, k, v))
        out = torch.empty_like(q)
        self._check(self.lib.cvk_op_attention(self.h, _ptr(q), _ptr(k), _ptr(v), _ints(lens), len(lens), heads, chunk, scale,
                                              _ptr(out), _stream()))
        return out

    # ------------------------------------------------------------------ HiFT
    def hift_f0(self, mel, lens):
        mel = _f32(mel, self.device)
        f0 = torch.empty(mel.shape[0], device=self.device)
        self._check(self.lib.cvk_hift_f0(self.h, _ptr(mel), _ints(lens), len(lens), _ptr(f0), _stream()))
        return f0

    def hift_source(self, f0, lens, noise):
        f0, noise = _f32(f0, self.device), _f32(noise, self.device)
        src = torch.empty(f0.shape[0] * 480, device=self.device)
        self._check(self.lib.cvk_hift_source(self.h, _ptr(f0), _ints(lens), len(lens), _ptr(noise), _ptr(src), _stream()))
        return src

    def hift_decode(self, mel, lens, source):
        mel, source = _f32(mel, self.device), _f32(source, self.device)
        wav = torch.empty(mel.shape[0] * 480, device=self.device)
        self._check(self.lib.cvk_hift_decode(self.h, _ptr(mel), _ints(lens), len(lens), _ptr(source), _ptr(wav), _stream()))
        return wav

    def hift_inference(self, mel, lens, noise, cache_source=None, cache_lens=None):
        mel, noise = _f32(mel, self.device), _f32(noise, self.device)
        wav = torch.empty(mel.shape[0] * 480, device=self.device)
        src = torch.empty(mel.shape[0] * 480, device=self.device)
        cs = _f32(cache_source, self.device) if cache_source is not None else None
        cl = _ints(cache_lens) if cache_lens is not None else None
        self._check(self.lib.cvk_hift_inference(self.h, _ptr(mel), _ints(lens), len(lens), _ptr(noise), _ptr(cs), cl, _ptr(wav),
                                                _ptr(src), _stream()))
        return wav, src

    # ------------------------------------------------------------------ flow
    def set_cfm_noise(self, noise_tm):
        noise_tm = _f32(noise_tm, self.device)
        self._check(self.lib.cvk_cfm_set_noise(self.h, _ptr(noise_tm), noise_tm.shape[0], 1))

    def flow_encoder(self, tokens, lens, streaming=False, context_len=0):
        tokens = tokens.to(device=self.device, dtype=torch.int32).contiguous()
        rows = sum(2 * (int(l) - context_len) for l in lens)
        h = torch.empty(rows, 512, device=self.device)
        self._check(self.lib.cvk_flow_encoder(self.h, _ptr(tokens), _ints(lens), len(lens), int(streaming), context_len, _ptr(h), _stream()))
        return h

    def cfm_estimator(self, x, mu, t, spks, cond, lens, streaming=False):
        x, mu, t, spks, cond = (_f32(a, self.device) for a in (x, mu, t, spks, cond))
        out = torch.empty_like(x)
        self._check(self.lib.cvk_cfm_estimator(self.h, _ptr(x), _ptr(mu), _ptr(t), _ptr(spks), _ptr(cond), _ints(lens), len(lens),
                                               int(streaming), _ptr(out), _stream()))
        return out

    def cfm_estimator_inplace(self, x, mu, t, spks, cond, lens, streaming=False):
        """the TensorRT engine contract (flow_matching.py:140-148): x [sum T, 80] float32 on the device is overwritten"""
        assert x.is_cuda and x.dtype == torch.float32 and x.is_contiguous()
        mu, t, spks, cond = (_f32(a, self.device) for a in (mu, t, spks, cond))
        self._check(self.lib.cvk_cfm_estimator_inplace(self.h, _ptr(x), _ptr(mu), _ptr(t), _ptr(spks), _ptr(cond), _ints(lens), len(lens),
                                                       int(streaming), _stream()))
        return x

    def workspace_bytes(self):
        cap, high = ctypes.c_size_t(), ctypes.c_size_t()
        self._check(self.lib.cvk_workspace_bytes(self.h, ctypes.byref(cap), ctypes.byref(high)))
        return cap.value, high.value

    def hift3_set_noise(self, rand_ini, sine_noise):
        """CosyVoice3 vocoder: SineGen2.rand_ini [9] and SineGen2.sine_waves [n,9] (module attributes of the reference)"""
        rand_ini = _f32(rand_ini.reshape(-1), self.device)
        sine_noise = _f32(sine_noise.reshape(-1, 9), self.device)
        self._check(self.lib.cvk_hift3_set_noise(self.h, _ptr(rand_ini), _ptr(sine_noise), sine_noise.shape[0], 1))

    def hift3_inference(self, mel, lens, finalize=True):
        """CausalHiFTGenerator.inference: mel [sum T, 80] -> (wav [sum 480 T], f0 [sum T], source [sum 480 T]); with finalize=False
        (streaming call) wav [sum 480 (T-8)], f0 [sum T-3], source [sum 480 (T-3)]"""
        mel = _f32(mel, self.device)
        # streaming call (finalize=False): 3 frames of f0 look-ahead, 4 of conv_pre look-ahead, the last frame's samples dropped
        n_src = sum(int(l) - (0 if finalize else 3) for l in lens)
        n_out = sum(int(l) - (0 if finalize else 8) for l in lens)
        wav = torch.empty(n_out * 480, device=self.device)
        f0 = torch.empty(n_src, device=self.device)
        src = torch.empty(n_src * 480, device=self.device)
        self._check(self.lib.cvk_hift3_inference(self.h, _ptr(mel), _ints(lens), len(lens), int(finalize), _ptr(wav), _ptr(f0), _ptr(src),
                                                 _stream()))
        return wav, f0, src

    def dit_estimator(self, x, mu, t, spks, cond, lens, streaming=False):
        """CosyVoice3 DiT estimator (stage "flow3"); same layout as cfm_estimator."""
        x, mu, t, spks, cond = (_f32(a, self.device) for a in (x, mu, t, spks, cond))
        out = torch.empty_like(x)
        self._check(self.lib.cvk_dit_estimator(self.h, _ptr(x), _ptr(mu), _ptr(t), _ptr(spks), _ptr(cond), _ints(lens), len(lens),
                                               int(streaming), _ptr(out), _stream()))
        return out

    def flow3_inference(self, tokens, token_lens, prompt_feat, prompt_feat_lens, embedding, n_timesteps=10, streaming=False,
                        finalize=True):
        """CosyVoice3 flow (CausalMaskedDiffWithDiT.inference); same layout as flow_inference."""
        tokens = tokens.to(device=self.device, dtype=torch.int32).contiguous()
        prompt_feat = _f32(prompt_feat, self.device) if prompt_feat is not None and prompt_feat.numel() else None
        embedding = _f32(embedding, self.device)
        ctxl = 0 if finalize else 3
        out_lens = [2 * (int(n) - ctxl) - int(p) for n, p in zip(token_lens, prompt_feat_lens)]
        mel = torch.empty(sum(out_lens), 80, device=self.device)
        self._check(self.lib.cvk_flow3_inference(self.h, _ptr(tokens), _ints(token_lens), _ptr(prompt_feat), _ints(prompt_feat_lens),
                                                 _ptr(embedding), len(token_lens), n_timesteps, int(streaming), int(finalize),
                                                 _ptr(mel), _stream()))
        return mel, out_lens

    def cfm_solve(self, mu, spks, cond, lens, z=None, n_timesteps=10, cfg_rate=0.7, streaming=False):
        mu, spks, cond = (_f32(a, self.device) for a in (mu, spks, cond))
        z = _f32(z, self.device) if z is not None else None
        out = torch.empty_like(mu)
        self._check(self.lib.cvk_cfm_solve(self.h, _ptr(mu), _ptr(spks), _ptr(cond), _ints(lens), len(lens), _ptr(z), n_timesteps,
                                           cfg_rate, int(streaming), _ptr(out), _stream()))
        return out

    def flow_inference(self, tokens, token_lens, prompt_feat, prompt_feat_lens, embedding, n_timesteps=10, streaming=False,
                       finalize=True):
        tokens = tokens.to(device=self.device, dtype=torch.int32).contiguous()
        prompt_feat = _f32(prompt_feat, self.device) if prompt_feat is not None and prompt_feat.numel() else None
        embedding = _f32(embedding, self.device)
        ctxl = 0 if finalize else 3
        out_lens = [2 * (int(n) - ctxl) - int(p) for n, p in zip(token_lens, prompt_feat_lens)]
        mel = torch.empty(sum(out_lens), 80, device=self.device)
        self._check(self.lib.cvk_flow_inference(self.h, _ptr(tokens), _ints(token_lens), _ptr(prompt_feat), _ints(prompt_feat_lens),
                                                _ptr(embedding), len(token_lens), n_timesteps, int(streaming), int(finalize),
                                                _ptr(mel), _stream()))
        return mel, out_lens

    # ------------------------------------------------------------------ incremental streaming flow (cvk.h: cvk_flow_stream_*)
    def flow_stream(self, max_frames, n_timesteps=10, dit=False):
        """dit=False: CosyVoice2 U-Net estimator (stage "flow"); dit=True: CosyVoice3 DiT (stage "flow3")"""
        s = ctypes.c_void_p()
        fn = self.lib.cvk_flow3_stream_create if dit else self.lib.cvk_flow_stream_create
        self._check(fn(self.h, int(max_frames), int(n_timesteps), ctypes.byref(s)))
        return s

    def flow_stream_destroy(self, fs):
        self.lib.cvk_flow_stream_destroy(self.h, fs)

    def flow_stream_bytes(self, fs):
        return int(self.lib.cvk_flow_stream_bytes(fs))

    def flow_stream_begin(self, fs, prompt_feat, embedding):
        """prompt_feat [Tp,80] (may be empty), embedding [192] or [1,192]"""
        pf = _f32(prompt_feat, self.device) if prompt_feat is not None and prompt_feat.numel() else None
        emb = _f32(embedding, self.device)
        self._check(self.lib.cvk_flow_stream_begin(self.h, fs, _ptr(pf), 0 if pf is None else int(pf.shape[0]), _ptr(emb), _stream()))

    def flow_stream_chunk(self, fs, tokens):
        """tokens: 1-D int32 = prompt tokens + speech tokens so far + 3 look-ahead tokens.  Returns the new mel frames [n,80]."""
        tokens = tokens.to(device=self.device, dtype=torch.int32).contiguous().reshape(-1)
        cap = 2 * int(tokens.numel())
        mel = torch.empty(cap, 80, device=self.device)
        n = ctypes.c_int(0)
        self._check(self.lib.cvk_flow_stream_chunk(self.h, fs, _ptr(tokens), int(tokens.numel()), _ptr(mel), cap, ctypes.byref(n), _stream()))
        return mel[:n.value]

    def flow_stream_slots(self, n_slots, max_frames, n_timesteps=10, dit=False):
        """One session holding n_slots utterances of up to max_frames mel frames each (cvk_flow_stream_slots_create)."""
        s = ctypes.c_void_p()
        self._check(self.lib.cvk_flow_stream_slots_create(self.h, int(bool(dit)), int(n_slots), int(max_frames), int(n_timesteps),
                                                          ctypes.byref(s)))
        return s

    def flow_stream_slot_begin(self, fs, slot, prompt_feat, embedding):
        """new utterance in `slot`: prompt_feat [Tp,80] (may be empty), embedding [192] or [1,192]"""
        pf = _f32(prompt_feat, self.device) if prompt_feat is not None and prompt_feat.numel() else None
        emb = _f32(embedding, self.device)
        self._check(self.lib.cvk_flow_stream_slot_begin(self.h, fs, int(slot), _ptr(pf), 0 if pf is None else int(pf.shape[0]), _ptr(emb),
                                                        _stream()))

    def flow_stream_chunk_batch(self, fs, slots, tokens_list):
        """Advance the distinct slots `slots` at once; tokens_list[b] = slot b's prompt tokens + speech tokens so far + 3
        look-ahead tokens.  Returns (new mel frames of every slot back to back [sum n, 80] on the device, n list)."""
        lens = [int(t.numel()) for t in tokens_list]
        tokens = torch.cat([t.reshape(-1).to(dtype=torch.int32) for t in tokens_list]).to(self.device).contiguous()
        cap = 2 * sum(lens)
        mel = torch.empty(cap, 80, device=self.device)
        n = (ctypes.c_int * len(lens))()
        self._check(self.lib.cvk_flow_stream_chunk_batch(self.h, fs, len(lens), _ints(slots), _ptr(tokens), _ints(lens), _ptr(mel), cap, n,
                                                         _stream()))
        n = list(n)
        return mel[:sum(n)], n

    # ------------------------------------------------------------------ LM
    def lm_session(self, max_batch, max_context):
        s = ctypes.c_void_p()
        self._check(self.lib.cvk_lm_session_create(self.h, max_batch, max_context, ctypes.byref(s)))
        return s

    def lm_session_destroy(self, s):
        self.lib.cvk_lm_session_destroy(self.h, s)

    def lm_prefill(self, sess, text, text_lens, speech, speech_lens):
        text = text.to(device=self.device, dtype=torch.int32).contiguous()
        speech = speech.to(device=self.device, dtype=torch.int32).contiguous()
        self._check(self.lib.cvk_lm_prefill(self.h, sess, _ptr(text), _ints(text_lens), _ptr(speech), _ints(speech_lens),
                                            len(text_lens), _stream()))

    def lm_decode(self, sess, n_steps, uniforms, min_len, max_len, out_ids, out_count, done, want_live=True):
        live = ctypes.c_int(0)
        self._check(self.lib.cvk_lm_decode(self.h, sess, n_steps, _ptr(uniforms), _ptr(min_len), _ptr(max_len), _ptr(out_ids),
                                           out_ids.shape[1], _ptr(out_count), _ptr(done),
                                           ctypes.byref(live) if want_live else None, _stream()))
        return live.value

    def lm_forward_logp(self, embeds, lens):
        embeds = _f32(embeds, self.device)
        out = torch.empty(embeds.shape[0], self.lm_vocab(), device=self.device)
        self._check(self.lib.cvk_lm_forward_logp(self.h, _ptr(embeds), _ints(lens), len(lens), _ptr(out), _stream()))
        return out

    def lm_vocab(self):
        """width of the LM's log-prob rows: 6564 (Qwen2LM) or 6764 (CosyVoice3LM, 3 impossible pad ids)"""
        return int(self.lib.cvk_lm_vocab(self.h))

    def lm_begin(self, sess, B=1):
        self._check(self.lib.cvk_lm_begin(self.h, sess, B, _stream()))

    def lm_feed(self, sess, ids, kinds):
        """ids / kinds: python int lists (kind 0 text id, 1 speech id, 2 llm_embedding row)"""
        self._check(self.lib.cvk_lm_feed(self.h, sess, _ints(ids), _ints(kinds), len(ids), _stream()))

    def lm_next_logp(self, sess, B=1):
        out = torch.empty(B, self.lm_vocab(), device=self.device)
        self._check(self.lib.cvk_lm_next_logp(self.h, sess, _ptr(out), _stream()))
        return out

    def lm_last_logits(self, sess, B):
        out = torch.empty(B, self.lm_vocab(), device=self.device)
        self._check(self.lib.cvk_lm_last_logits(self.h, sess, _ptr(out), _stream()))
        return out

    def ras_sample(self, logp, history, hist_count, uniforms, ignore_eos):
        logp = _f32(logp, self.device).clone()
        history = history.to(device=self.device, dtype=torch.int32).contiguous()
        hist_count = hist_count.to(device=self.device, dtype=torch.int32).contiguous()
        uniforms = _f32(uniforms, self.device)
        ignore_eos = ignore_eos.to(device=self.device, dtype=torch.int32).contiguous()
        out = torch.empty(logp.shape[0], dtype=torch.int32, device=self.device)
        self._check(self.lib.cvk_ras_sample(self.h, _ptr(logp), logp.shape[0], logp.shape[1], _ptr(history), history.shape[1],
                                            _ptr(hist_count), _ptr(uniforms), _ptr(ignore_eos), _ptr(out), _stream()))
        return out

    # ------------------------------------------------------------------ mel
    def whisper_log_mel(self, wav, lens):
        """wav [sum N_b] at 16 kHz -> [sum N_b // 160, 128] (whisper.log_mel_spectrogram(n_mels=128), time-major)"""
        wav = _f32(wav, self.device)
        out = torch.empty(sum(int(l) // 160 for l in lens), 128, device=self.device)
        self._check(self.lib.cvk_whisper_log_mel(self.h, _ptr(wav), _ints(lens), len(lens), _ptr(out), _stream()))
        return out

    def kaldi_fbank(self, wav, lens, subtract_mean=True):
        """wav [sum N_b] at 16 kHz -> [sum 1 + (N_b - 400) // 160, 80] (kaldi.fbank(num_mel_bins=80, dither=0) [- mean over frames])"""
        wav = _f32(wav, self.device)
        out = torch.empty(sum(1 + (int(l) - 400) // 160 for l in lens), 80, device=self.device)
        self._check(self.lib.cvk_kaldi_fbank(self.h, _ptr(wav), _ints(lens), len(lens), int(bool(subtract_mean)), _ptr(out), _stream()))
        return out

    def mel_spectrogram(self, wav, lens, fmax=8000):
        """wav [sum N_b] -> mel [sum N_b // 480, 80]; fmax 8000 (CosyVoice2) or None / 12000 (CosyVoice3)"""
        wav = _f32(wav, self.device)
        mel = torch.empty(sum(int(l) // 480 for l in lens), 80, device=self.device)
        self._check(self.lib.cvk_mel_spectrogram_ex(self.h, _ptr(wav), _ints(lens), len(lens), int(fmax or 0), _ptr(mel), _stream()))
        return mel
