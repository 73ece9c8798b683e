"""Host-side mirror of the reference pipeline orchestrator, over libcvk.

``B200CosyVoice2Model`` exposes the constructor / ``load`` / ``tts`` / ``token2wav`` surface and the session attributes
of ``cosyvoice.cli.model.CosyVoice2Model`` (cosyvoice/cli/model.py:245-394) so it can be dropped in behind
``cosyvoice.cli.cosyvoice.CosyVoice2`` (``cosyvoice.model = B200CosyVoice2Model(...)``, see INTEGRATION.md), plus
``tts_batch`` for the batch-32 metric (the reference has no batched API; its batch is a Python loop).

All arithmetic happens in libcvk (hand-written sm_100a kernels); torch provides device memory, streams and the two
random streams the reference draws from the global RNG (sampling uniforms, SineGen noise).  No CPU fallback.
"""
import threading
import time
import uuid
from contextlib import nullcontext

import numpy as np
import torch

from . import cvk

TOKEN_MEL_RATIO = 2          # cosyvoice2.yaml:14
PRE_LOOKAHEAD = 3            # cosyvoice2.yaml:46
SAMPLES_PER_FRAME = 480


def _count(keys, prefix):
    idx = set()
    for k in keys:
        if k.startswith(prefix):
            idx.add(int(k[len(prefix):].split(".")[0]))
    return len(idx)


def infer_cfgs(llm_sd, flow_sd):
    """layer counts from state_dict keys (the reference builds these from yaml; cosyvoice2.yaml:23-87)"""
    nl = _count(llm_sd.keys(), "llm.model.model.layers.")
    fk = list(flow_sd.keys())
    flow_cfg = [_count(fk, "encoder.encoders."), _count(fk, "encoder.up_encoders."), _count(fk, "decoder.estimator.mid_blocks."),
                _count(fk, "decoder.estimator.down_blocks.0.1.")]
    return [nl], flow_cfg


def _state_dict(m):
    return m if isinstance(m, dict) else m.state_dict()


def cfm_rand_noise():
    """CausalConditionalCFM.rand_noise (flow/flow_matching.py:199-200): seed-0 torch.randn([1,80,15000]), time-major."""
    g = torch.Generator(device="cpu")
    g.manual_seed(0)
    return torch.randn([1, 80, 50 * 300], generator=g)[0].t().contiguous()


class B200CosyVoice2Model:
    # text-streaming LM constants: Qwen2LM (llm.py:275-277: eos = speech_token_size, fill = speech_token_size + 2, whole
    # prompt text goes into the text cache).  B200CosyVoice3Model overrides them (CosyVoice3LM, llm.py:681-684, 583-588).
    bistream_fill_token = 6563
    bistream_eos_token = 6561
    bistream_eop_token = None
    # benchmark aid only (None = the reference's behaviour: decode "until met eos", llm.py:642-661, without any cap): random-init
    # weights cannot be made to emit eos at a chosen time, so bench.py ends the text-streaming decode after this many ids
    bistream_max_tokens = None
    # streaming synthesis: intermediate chunks through the cached flow session (cvk_flow_stream_*: each chunk computes only its new
    # frames) instead of the reference's prefix recompute (cli/model.py:346-363); same frames either way.  The U-Net estimator of
    # B200CosyVoice3Model uses the same sessions for its DiT.
    incremental_flow = True
    flow_stream_dit = False              # which estimator the sessions cache: the CosyVoice2 U-Net (stage "flow") or the CosyVoice3 DiT ("flow3")
    stream_cache_frames = 2048           # mel frames (prompt included) one streaming request can cache (41 s); ~2.3 MB per frame in bf16

    def __init__(self, llm=None, flow=None, hift=None, fp16=False, precision="bf16", device=0, workspace_gb=24.0):
        # attribute names follow cli/model.py:245-275
        self.device = torch.device("cuda", device)
        self.llm, self.flow, self.hift = llm, flow, hift
        self.fp16 = fp16
        self.token_hop_len = 25
        self.token_max_hop_len = 4 * self.token_hop_len
        self.stream_scale_factor = 2
        self.mel_cache_len = 8
        self.source_cache_len = int(self.mel_cache_len * 480)
        self.speech_window = np.hamming(2 * self.source_cache_len)
        self.lock = threading.Lock()
        self.tts_speech_token_dict = {}
        self.llm_end_dict = {}
        self.hift_cache_dict = {}
        self.silent_tokens = []
        self.ctx = cvk.Context(device, precision, workspace_gb)
        self.stream = torch.cuda.Stream(self.device)     # every library call of this model runs on this stream
        self.generator = torch.Generator(device=self.device)
        self.generator.manual_seed(1986)
        self._free_sessions = {}             # (B, ctx rounded to 256) -> idle cvk_lm_session handles (see _checkout_session)
        self._session_lru = []               # keys of idle sessions, least recently returned first
        self.max_idle_sessions = 4
        self._pool_lock = threading.Lock()
        self._lm_streams = []
        self.flow_stream_dict = {}           # uuid -> cvk_flow_stream handle, or False once a request has left the chunk grid
        self._idle_flow_streams = []
        self._idle_slot_session = None       # ((dit, n_slots, cap), cvk_flow_stream handle) kept by tts_stream_batch
        self.lm_chains = 1                   # independent decode chains run concurrently (see lm_generate)
        self._window = torch.from_numpy(self.speech_window).float().to(self.device)
        self.n_timesteps = 10
        self.min_token_text_ratio, self.max_token_text_ratio = 2.0, 20.0
        self.timings = {}
        # test hooks: explicit random streams instead of the device generator (the reference uses the global torch RNG)
        self.uniforms_override = None        # tensor [steps, B, 2]
        self.noise_fn = None                 # callable(n_samples) -> [n_samples, 9]
        if llm is not None and flow is not None and hift is not None:
            self.load_state_dicts(_state_dict(llm), _state_dict(flow), _state_dict(hift))

    # ---------------------------------------------------------------- weights (cli/model.py:65-73)
    def load(self, llm_model, flow_model, hift_model):
        llm_sd = torch.load(llm_model, map_location="cpu", weights_only=True)
        flow_sd = torch.load(flow_model, map_location="cpu", weights_only=True)
        hift_sd = {k.replace("generator.", ""): v for k, v in torch.load(hift_model, map_location="cpu", weights_only=True).items()}
        self.load_state_dicts(llm_sd, flow_sd, hift_sd)

    def load_state_dicts(self, llm_sd, flow_sd, hift_sd):
        llm_cfg, flow_cfg = infer_cfgs(llm_sd, flow_sd)
        self.ctx.load_state_dict("llm", llm_sd, llm_cfg)
        self.ctx.load_state_dict("flow", flow_sd, flow_cfg)
        self.ctx.load_state_dict("hift", hift_sd)
        self.ctx.set_cfm_noise(cfm_rand_noise())
        self.ctx.finalize("mel")

    # engine swap points of the reference are meaningless here; kept so that CosyVoice2.__init__ flags fail loudly
    def load_jit(self, *a, **k):
        raise RuntimeError("B200CosyVoice2Model has no TorchScript path (cli/model.py:277-279 swap point is replaced by libcvk)")

    def load_trt(self, *a, **k):
        raise RuntimeError("B200CosyVoice2Model has no TensorRT path (the estimator runs in libcvk)")

    def load_vllm(self, *a, **k):
        raise RuntimeError("B200CosyVoice2Model has no vLLM path (the LM runs in libcvk)")

    # ---------------------------------------------------------------- LM (llm/llm.py:458-549), batched
    def _checkout_session(self, B, ctx_len):
        """An LM session (KV cache + decode buffers + captured step graph) is owned by ONE generation from prefill to the last
        token: the reference keeps per-request state keyed by uuid (cli/model.py:334-337) and serves overlapping tts() calls
        from threads, so two requests of similar shape must never share a KV cache.  Idle sessions are kept for re-use
        (creating one allocates hundreds of MB at batch 32) and the idle pool is bounded (LRU, cvk_lm_session_destroy)."""
        key = (B, (ctx_len + 255) // 256 * 256)
        with self._pool_lock:
            free = self._free_sessions.get(key)
            if free:
                self._session_lru.remove(key)
                return key, free.pop()
        return key, self.ctx.lm_session(*key)

    def _new_lm_stream(self):
        return torch.cuda.Stream(self.device) if self.device.type == "cuda" else None

    def _checkin_session(self, key, sess):
        evict = []
        with self._pool_lock:
            self._free_sessions.setdefault(key, []).append(sess)
            self._session_lru.append(key)
            while len(self._session_lru) > self.max_idle_sessions:
                k = self._session_lru.pop(0)
                evict.append(self._free_sessions[k].pop(0))
        for e in evict:
            self.ctx.lm_session_destroy(e)

    def lm_generate(self, texts, prompt_texts, prompt_speech_tokens, uniforms=None, steps_per_sync=32, on_progress=None, stream=None):
        """texts/prompt_texts/prompt_speech_tokens: lists of int32 tensors [1,n].  Returns a list of python id lists.

        `stream`: CUDA stream for this generation (default: the model's stream).  Only the prefill uses the shared workspace and
        takes `ctx.lock`; the decode calls touch nothing but their own session (include/cvk.h threading rules), so a request's
        LM job on its own stream overlaps another request's - or its own - flow / vocoder calls like the reference's LM thread
        does (cli/model.py:101-129, 268).

        `self.lm_chains > 1` splits the rows into independent groups, each with its own KV session, CUDA graph and stream (an
        experiment knob from the per-op decode chain; with the persistent decode kernel one chain is best).  Results are
        independent of the grouping (rows never interact; every row consumes its own uniforms)."""
        B = len(texts)
        d = self.device
        main = stream if stream is not None else self.stream
        chains = 1 if on_progress is not None else max(1, min(self.lm_chains, B))
        groups = [list(range(g, B, chains)) for g in range(chains)]
        mins = [int(t.shape[1] * self.min_token_text_ratio) for t in texts]      # llm.py:497-498
        maxs = [int(t.shape[1] * self.max_token_text_ratio) for t in texts]
        mx = max(maxs)
        st = []
        try:
            # The prefill uses the context's shared workspace arena, so it runs on the model's stream under ctx.lock like every other
            # workspace call (flow / vocoder): the lock orders the host calls, the common stream orders the device work.  Only the
            # decode steps - which touch nothing but their session - run on the generation's own stream.
            with torch.cuda.stream(self.stream):
                if uniforms is None and self.uniforms_override is not None:
                    uniforms = self.uniforms_override
                if uniforms is None:
                    with self.lock:                                  # one device generator shared by the request threads
                        uniforms = torch.rand(mx + 1, B, 2, device=d, generator=self.generator)
                uniforms = uniforms.to(d).float()
                for g, rows in enumerate(groups):
                    tl = [int(texts[r].shape[1] + prompt_texts[r].shape[1]) for r in rows]
                    sl = [int(prompt_speech_tokens[r].shape[1]) for r in rows]
                    tt = torch.cat([torch.cat([prompt_texts[r].reshape(-1).to(d, non_blocking=True), texts[r].reshape(-1).to(d, non_blocking=True)])
                                    for r in rows]).to(torch.int32)
                    ss = torch.cat([prompt_speech_tokens[r].reshape(-1).to(d, non_blocking=True) for r in rows]).to(torch.int32) if sum(sl) \
                        else torch.zeros(1, dtype=torch.int32, device=d)
                    key, sess = self._checkout_session(len(rows), max(a + b2 for a, b2 in zip(tl, sl)) + 2 + mx + 8)
                    c = dict(rows=rows, n=len(rows), key=key, sess=sess,
                             min_len=torch.tensor([mins[r] for r in rows], dtype=torch.int32, device=d),
                             max_len=torch.tensor([maxs[r] for r in rows], dtype=torch.int32, device=d),
                             max_len_host=torch.tensor([maxs[r] for r in rows], dtype=torch.int32),
                             out_ids=torch.zeros(len(rows), mx + 1, dtype=torch.int32, device=d),
                             out_count=torch.zeros(len(rows), dtype=torch.int32, device=d),
                             done=torch.zeros(len(rows), dtype=torch.int32, device=d),
                             U=uniforms[:, rows, :].contiguous(), live=len(rows))
                    st.append(c)
                    with self.ctx.lock:
                        self.ctx.lm_prefill(sess, tt, tl, ss, sl)
                        ready = torch.cuda.Event()
                        ready.record(self.stream)
                    c["ready"] = ready
            while len(self._lm_streams) < chains:
                self._lm_streams.append(torch.cuda.Stream(d))
            n = 0
            for c in st:
                c["left"] = mx                     # upper bound of the steps this chain still needs (refined after every block)
            while True:
                for g, c in enumerate(st):
                    if c["live"] == 0:
                        continue
                    s_g = main if chains == 1 else self._lm_streams[g]
                    with torch.cuda.stream(s_g):
                        if n == 0:
                            s_g.wait_event(c["ready"])
                        # never run past the longest possible remainder: the last block is cut to what the live rows can still emit
                        # (round 1 always ran whole blocks: 320 steps for rows that end at 300)
                        c["block"] = max(1, min(steps_per_sync, c["left"]))
                        self.ctx.lm_decode(c["sess"], c["block"], c["U"], c["min_len"], c["max_len"], c["out_ids"], c["out_count"], c["done"],
                                           want_live=False)
                for g, c in enumerate(st):
                    if c["live"] == 0:
                        continue
                    s_g = main if chains == 1 else self._lm_streams[g]
                    with torch.cuda.stream(s_g):
                        c["live"] = self.ctx.lm_decode(c["sess"], 0, c["U"], c["min_len"], c["max_len"], c["out_ids"], c["out_count"], c["done"])
                        if c["live"]:
                            cnt, dn = c["out_count"].cpu(), c["done"].cpu()
                            c["left"] = int(((c["max_len_host"] - cnt) * (dn == 0)).max())
                n += steps_per_sync
                if on_progress is not None:
                    on_progress(st[0]["out_ids"], st[0]["out_count"], st[0]["live"], st[0]["done"])
                if all(c["live"] == 0 for c in st) or n > mx + steps_per_sync:
                    break
            out = [None] * B
            for g, c in enumerate(st):
                with torch.cuda.stream(main if chains == 1 else self._lm_streams[g]):
                    cnt = c["out_count"].cpu().tolist()
                    ids = c["out_ids"].cpu()
                for i, r in enumerate(c["rows"]):
                    out[r] = ids[i, :cnt[i]].tolist()
            if chains > 1:
                for g in range(chains):
                    main.wait_stream(self._lm_streams[g])
            return out
        finally:
            main.synchronize()                     # the session goes back to the pool only when its last kernel has finished
            for c in st:
                self._checkin_session(c["key"], c["sess"])

    def lm_generate_bistream(self, text, prompt_text, prompt_speech_token, uniforms=None, stream=None):
        """llm/llm.py:551-661 (Qwen2LM.inference_bistream): `text` is a generator of int32 [1,k] chunks; speech ids are yielded
        as soon as they are decoded.  The interleaving (5 text : 15 speech), the forced / sampled fill tokens and the final
        'decode until eos' phase are the reference's control flow line for line; the arithmetic runs on the device through
        cvk_lm_begin / cvk_lm_feed / cvk_lm_next_logp / cvk_ras_sample.  uniforms [n,2]: row len(out_tokens) is consumed by the
        draw that produces that token (default: drawn from the model's generator)."""
        mix_text, mix_speech = 5, 15
        fill_token, eos_token, speech_vocab = self.bistream_fill_token, self.bistream_eos_token, 6561
        TEXT, SPEECH, LLM = 0, 1, 2
        d = self.device
        ptext = [int(x) for x in prompt_text.reshape(-1).tolist()]
        lm_prefix = []
        if self.bistream_eop_token is not None:
            # llm.py:583-588: the prompt text up to and including <|endofprompt|> is fed ahead of the 5:15 interleaving
            if self.bistream_eop_token not in ptext:
                raise AssertionError("<|endofprompt|> not detected in CosyVoice3 prompt_text, check your input!")
            eop = ptext.index(self.bistream_eop_token)
            lm_prefix, ptext = [(TEXT, t) for t in ptext[:eop + 1]], ptext[eop + 1:]
        pspeech = [int(x) for x in prompt_speech_token.reshape(-1).tolist()]
        max_ctx = 4096
        lm_stream = stream if stream is not None else self.stream
        key, sess = self._checkout_session(1, max_ctx - 8)
        with torch.cuda.stream(lm_stream):
            self.ctx.lm_begin(sess, 1)
        if uniforms is None and self.uniforms_override is not None:
            uniforms = self.uniforms_override[:, 0, :]
        # `lm_input` has the reference variable's exact life cycle (list of (kind, id) positions): every model call pushes ALL
        # of it, it is replaced after a yielded token and - like the reference - left untouched when a fill token ends a decode
        # burst, so a final phase entered right after a fill token pushes that last input a second time (llm.py:634-637, 643).
        lm_input = [(LLM, 0)] + lm_prefix
        text_cache = list(ptext)
        out_tokens = []
        next_fill_index = (len(pspeech) // mix_speech + 1) * mix_speech - len(pspeech)
        fed = [0]

        def forward(want_logp):
            """llm.py:617-622: push lm_input through the cached model; log-probs of the next id"""
            with torch.cuda.stream(lm_stream):
                fed[0] += len(lm_input)
                if fed[0] >= max_ctx - 16:
                    raise RuntimeError("text-streaming LM: session context exhausted")
                self.ctx.lm_feed(sess, [i for _, i in lm_input], [k for k, _ in lm_input])
                return self.ctx.lm_next_logp(sess, 1) if want_logp else None

        def sample(logp, ignore_eos):
            """llm.py:627 / 650 sampling_ids"""
            with torch.cuda.stream(lm_stream):
                i = len(out_tokens)
                if uniforms is not None:
                    u = uniforms[i].reshape(1, 2)
                else:
                    with self.lock:
                        u = torch.rand(1, 2, device=d, generator=self.generator)
                hist = torch.tensor([out_tokens[-16:] or [0]], dtype=torch.int32)
                top = self.ctx.ras_sample(logp, hist, torch.tensor([min(len(out_tokens), 16)], dtype=torch.int32), u,
                                          torch.tensor([1 if ignore_eos else 0], dtype=torch.int32))
                return int(top.item())

        try:
            for this_text in text:
                text_cache += [int(x) for x in this_text.reshape(-1).tolist()]
                while pspeech:                                            # llm.py:595-604
                    if len(text_cache) >= mix_text:
                        lm_input = lm_input + [(TEXT, t) for t in text_cache[:mix_text]] + [(SPEECH, t) for t in pspeech[:mix_speech]]
                        text_cache, pspeech = text_cache[mix_text:], pspeech[mix_speech:]
                    else:
                        break
                if not pspeech:                                           # llm.py:606-640
                    if (out_tokens and out_tokens[-1] == fill_token) or (not out_tokens and len(lm_input) == 1):
                        if len(text_cache) >= mix_text:
                            lm_text = [(TEXT, t) for t in text_cache[:mix_text]]
                            lm_input = lm_text if (out_tokens and out_tokens[-1] == fill_token) else lm_input + lm_text
                            text_cache = text_cache[mix_text:]
                        else:
                            continue
                    while True:
                        forced = next_fill_index != -1 and len(out_tokens) == next_fill_index
                        logp = forward(want_logp=not forced)              # the reference runs the model before overriding the draw
                        if forced:
                            top = fill_token
                            next_fill_index += mix_speech + 1
                        else:
                            top = sample(logp, ignore_eos=True)
                        if top == fill_token:
                            next_fill_index = len(out_tokens) + mix_speech + 1
                        out_tokens.append(top)
                        if top >= speech_vocab:
                            if top == fill_token:
                                break
                            raise ValueError(f"should not get token {top}")
                        yield top
                        lm_input = [(SPEECH, top)]
            lm_input = lm_input + [(TEXT, t) for t in text_cache] + [(LLM, 1)]       # llm.py:643
            while True:
                if self.bistream_max_tokens is not None and len(out_tokens) >= self.bistream_max_tokens:
                    break
                top = sample(forward(want_logp=True), ignore_eos=False)
                out_tokens.append(top)
                if top >= speech_vocab:
                    if top == eos_token:
                        break
                    raise ValueError(f"should not get token {top}")
                yield top
                lm_input = [(SPEECH, top)]
        finally:
            if lm_stream is not None:
                lm_stream.synchronize()
            self._checkin_session(key, sess)

    # ---------------------------------------------------------------- flow + vocoder
    def flow_batch(self, tokens, prompt_tokens, prompt_feats, embeddings, streaming=False, finalize=True):
        """lists per utterance: tokens [1,N] int, prompt_tokens [1,P], prompt_feats [1,Tp,80], embeddings [1,192]
        -> (mel [sum T,80] time-major on the device, lens)"""
        d = self.device
        tl = [int(t.shape[1] + p.shape[1]) for t, p in zip(tokens, prompt_tokens)]
        pl = [int(f.shape[1]) for f in prompt_feats]
        with torch.cuda.stream(self.stream), self.ctx.lock:
            toks = torch.cat([torch.cat([p.reshape(-1).to(d, non_blocking=True), t.reshape(-1).to(d, non_blocking=True)])
                              for t, p in zip(tokens, prompt_tokens)]).to(torch.int32)
            pf = torch.cat([f[0].to(d, non_blocking=True) for f in prompt_feats], 0) if sum(pl) else None
            emb = torch.cat([e.reshape(1, -1).to(d, non_blocking=True) for e in embeddings], 0)
            return self.ctx.flow_inference(toks, tl, pf, pl, emb, n_timesteps=self.n_timesteps, streaming=streaming, finalize=finalize)

    def hift_batch(self, mel_tm, lens, cache_source=None, cache_lens=None, noise=None):
        with torch.cuda.stream(self.stream), self.ctx.lock:
            if noise is None and self.noise_fn is not None:
                noise = self.noise_fn(sum(lens) * SAMPLES_PER_FRAME)
            if noise is None:
                noise = torch.randn(sum(lens) * SAMPLES_PER_FRAME, 9, device=self.device, generator=self.generator)
            return self.ctx.hift_inference(mel_tm, lens, noise, cache_source, cache_lens)

    def tts_batch_device(self, inputs, uniforms=None, noise=None):
        """The batched pipeline with the result left on the device: returns (wav_flat, lens, stats) - wav_flat is the vocoder's
        output buffer (float32 [sum n_i], the utterances back to back in input order, empty ones skipped), lens[i] the sample
        count of input i (0 when the LM produced no token).  Used by tts_batch and by the multi-GPU gather (parallel.gather_flat)."""
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        with torch.cuda.stream(self.stream):
            ev[0].record()
        ids = self.lm_generate([i["text"] for i in inputs], [i["prompt_text"] for i in inputs],
                               [i["llm_prompt_speech_token"] for i in inputs], uniforms)
        with torch.cuda.stream(self.stream):
            ev[1].record()
        toks = [torch.tensor(x, dtype=torch.int32).unsqueeze(0) for x in ids]
        keep = [b for b, x in enumerate(ids) if len(x) > 0]
        mel, lens = self.flow_batch([toks[b] for b in keep], [inputs[b]["flow_prompt_speech_token"] for b in keep],
                                    [inputs[b]["prompt_speech_feat"] for b in keep], [inputs[b]["flow_embedding"] for b in keep])
        with torch.cuda.stream(self.stream):
            ev[2].record()
        wav, _ = self.hift_batch(mel, lens, noise=noise)
        with torch.cuda.stream(self.stream):
            ev[3].record()
        n = [0] * len(inputs)
        for b, L in zip(keep, lens):
            n[b] = L * SAMPLES_PER_FRAME
        stats = {"ev": ev, "tokens": [len(x) for x in ids], "mel_frames": lens}
        return wav, n, stats

    def _stage_ms(self, stats):
        ev = stats.pop("ev")
        stats.update({"lm_ms": ev[0].elapsed_time(ev[1]), "flow_ms": ev[1].elapsed_time(ev[2]), "hift_ms": ev[2].elapsed_time(ev[3])})
        return stats

    def tts_batch(self, inputs, uniforms=None, noise=None, return_stats=False, to_host=True):
        """inputs: list of dicts with the kwargs of tts() (text, prompt_text, llm_prompt_speech_token,
        flow_prompt_speech_token, prompt_speech_feat, flow_embedding).  Returns a list of waveforms [1,N]
        (CPU tensors, or views of one device buffer when to_host=False)."""
        wav, n, stats = self.tts_batch_device(inputs, uniforms, noise)
        with torch.cuda.stream(self.stream):
            host = wav.cpu() if to_host else wav          # one D2H for the whole batch
        self.stream.synchronize()
        out, o = [], 0
        for k in n:
            out.append(host[o:o + k].unsqueeze(0) if k else torch.zeros(1, 0))
            o += k
        self.timings = self._stage_ms(stats)
        return (out, dict(self.timings)) if return_stats else out

    # ---------------------------------------------------------------- reference-shaped single-request API
    def _fade_in_out(self, fade_in, fade_out):
        """utils/common.py:170-178 without the CPU round trip."""
        n = self.source_cache_len
        fade_in = fade_in.clone()
        fade_in[..., :n] = fade_in[..., :n] * self._window[:n] + fade_out[..., -n:] * self._window[n:]
        return fade_in

    def _to_host(self, t):
        """D2H on the model's stream (the kernels that produced `t` were enqueued there, not on torch's current stream)."""
        with torch.cuda.stream(self.stream):
            h = t.cpu()
        self.stream.synchronize()
        return h

    def _flow_stream_chunk(self, token, prompt_token, prompt_feat, embedding, token_offset, uuid):
        """The frames of this streaming chunk from the request's cached flow session, or None when the request cannot use one
        (chunk ends off the 50-frame grid, prompt mel not 2 frames per prompt token, longer than the cache): the caller then
        recomputes the prefix like the reference."""
        if not self.incremental_flow or uuid not in self.tts_speech_token_dict:
            return None
        fs = self.flow_stream_dict.get(uuid)
        if fs is False:
            return None
        P = int(prompt_token.shape[1])
        total = TOKEN_MEL_RATIO * (P + int(token.shape[1]) - PRE_LOOKAHEAD)
        done = TOKEN_MEL_RATIO * (P + token_offset) if token_offset else 0
        chunk = 2 * 25                                   # cosyvoice2.yaml:16 static_chunk_size x token_mel_ratio
        ok = (total % chunk == 0 and done % chunk == 0 and int(prompt_feat.shape[1]) == TOKEN_MEL_RATIO * P
              and total <= self.stream_cache_frames and (fs is not None or token_offset == 0))
        if not ok:
            if fs:
                self._release_flow_stream(uuid)
            self.flow_stream_dict[uuid] = False
            return None
        d = self.device
        with torch.cuda.stream(self.stream), self.ctx.lock:
            if fs is None:
                with self._pool_lock:
                    fs = self._idle_flow_streams.pop() if self._idle_flow_streams else None
                if fs is None:
                    try:
                        fs = self.ctx.flow_stream(self.stream_cache_frames, self.n_timesteps, dit=self.flow_stream_dit)
                    except cvk.CvkError:
                        # no memory for another session's caches (several GB each): this request recomputes the prefix like the reference
                        self.flow_stream_dict[uuid] = False
                        return None
                self.flow_stream_dict[uuid] = fs
                self.ctx.flow_stream_begin(fs, prompt_feat[0].to(d, non_blocking=True), embedding.reshape(-1).to(d, non_blocking=True))
            toks = torch.cat([prompt_token.reshape(-1).to(d, non_blocking=True), token.reshape(-1).to(d, non_blocking=True)]).to(torch.int32)
            return self.ctx.flow_stream_chunk(fs, toks)

    def _release_flow_stream(self, uuid):
        fs = self.flow_stream_dict.pop(uuid, None)
        if fs:
            with self._pool_lock:
                if len(self._idle_flow_streams) < 2:
                    self._idle_flow_streams.append(fs)
                    fs = None
            if fs:
                self.stream.synchronize()
                self.ctx.flow_stream_destroy(fs)

    def token2wav(self, token, prompt_token, prompt_feat, embedding, token_offset, uuid, stream=False, finalize=False, speed=1.0):
        """cli/model.py:292-326"""
        new_mel = self._flow_stream_chunk(token.to(torch.int32), prompt_token, prompt_feat, embedding, token_offset, uuid) \
            if (stream and not finalize) else None
        if new_mel is None:
            mel, lens = self.flow_batch([token.to(torch.int32)], [prompt_token], [prompt_feat], [embedding], streaming=stream, finalize=finalize)
        with torch.cuda.stream(self.stream):
            tts_mel = new_mel if new_mel is not None else mel[token_offset * TOKEN_MEL_RATIO:]
            cache = self.hift_cache_dict[uuid]
            cache_source, cache_lens = None, None
            if cache is not None:
                tts_mel = torch.cat([cache["mel"], tts_mel], 0)
                cache_source, cache_lens = cache["source"], [cache["source"].shape[0]]
            if finalize is False:
                wav, src = self.hift_batch(tts_mel.contiguous(), [tts_mel.shape[0]], cache_source, cache_lens)
                if cache is not None:
                    wav = self._fade_in_out(wav, cache["speech"])
                self.hift_cache_dict[uuid] = {"mel": tts_mel[-self.mel_cache_len:].clone(), "source": src[-self.source_cache_len:].clone(),
                                              "speech": wav[-self.source_cache_len:].clone()}
                wav = wav[:-self.source_cache_len]
            else:
                if speed != 1.0:
                    assert cache is None, "speed change only support non-stream inference mode"
                    m = torch.nn.functional.interpolate(tts_mel.t().unsqueeze(0), size=int(tts_mel.shape[0] / speed), mode="linear")
                    tts_mel = m[0].t()
                wav, src = self.hift_batch(tts_mel.contiguous(), [tts_mel.shape[0]], cache_source, cache_lens)
                if cache is not None:
                    wav = self._fade_in_out(wav, cache["speech"])
        return wav.unsqueeze(0)

    def llm_job(self, text, prompt_text, llm_prompt_speech_token, llm_embedding, uuid):
        """cli/model.py:101-129 (non-generator text).  Tokens are appended to the session list as they arrive."""
        if hasattr(text, "__next__") or (hasattr(text, "__iter__") and not torch.is_tensor(text)):
            # cli/model.py:113-123: text generator -> bi-stream decoding, tokens appended one by one
            cur_silent, max_silent = 0, 5                  # cli/model.py:102,121-127 (silent_tokens is empty for CosyVoice2)
            for tok in self.lm_generate_bistream(iter(text), prompt_text, llm_prompt_speech_token, stream=self._new_lm_stream()):
                if tok in self.silent_tokens:
                    cur_silent += 1
                    if cur_silent > max_silent:
                        continue
                else:
                    cur_silent = 0
                self.tts_speech_token_dict[uuid].append(tok)
            self.llm_end_dict[uuid] = True
            return

        st = {"consumed": 0, "silent": 0}

        def progress(out_ids, out_count, live, done):
            self._take_tokens(out_ids[0], int(out_count[0].item()), st, self.tts_speech_token_dict[uuid])
        # the LM job decodes on its own stream (cli/model.py:103: `with self.llm_context`, a side stream) while token2wav runs on
        # the model's stream
        self.lm_generate([text], [prompt_text], [llm_prompt_speech_token], steps_per_sync=8, on_progress=progress,
                         stream=self._new_lm_stream())
        self.llm_end_dict[uuid] = True

    def _take_tokens(self, out_ids, n, st, dst):
        """append ids [st["consumed"], n) of one LM row to dst, dropping silent tokens past 5 in a row (cli/model.py:121-127;
        an empty list for CosyVoice2: never taken)"""
        if n > st["consumed"]:
            for tok in out_ids[st["consumed"]:n].tolist():
                if tok in self.silent_tokens:
                    st["silent"] += 1
                    if st["silent"] > 5:
                        continue
                else:
                    st["silent"] = 0
                dst.append(tok)
            st["consumed"] = n

    def vc_job(self, source_speech_token, uuid):
        self.tts_speech_token_dict[uuid] = source_speech_token.flatten().tolist()
        self.llm_end_dict[uuid] = True

    def tts(self, text=torch.zeros(1, 0, dtype=torch.int32), flow_embedding=torch.zeros(0, 192), llm_embedding=torch.zeros(0, 192),
            prompt_text=torch.zeros(1, 0, dtype=torch.int32), llm_prompt_speech_token=torch.zeros(1, 0, dtype=torch.int32),
            flow_prompt_speech_token=torch.zeros(1, 0, dtype=torch.int32), prompt_speech_feat=torch.zeros(1, 0, 80),
            source_speech_token=torch.zeros(1, 0, dtype=torch.int32), stream=False, speed=1.0, **kwargs):
        """cli/model.py:328-394: same signature, same yielded dicts ({'tts_speech': float32 CPU [1,N]})."""
        this_uuid = str(uuid.uuid1())
        with self.lock:
            self.tts_speech_token_dict[this_uuid], self.llm_end_dict[this_uuid] = [], False
            self.hift_cache_dict[this_uuid] = None
        if source_speech_token.shape[1] == 0:
            p = threading.Thread(target=self.llm_job, args=(text, prompt_text, llm_prompt_speech_token, llm_embedding, this_uuid))
        else:
            p = threading.Thread(target=self.vc_job, args=(source_speech_token, this_uuid))
        p.start()
        if stream is True:
            token_offset = 0
            P = flow_prompt_speech_token.shape[1]
            prompt_token_pad = int(np.ceil(P / self.token_hop_len) * self.token_hop_len - P)
            while True:
                time.sleep(0.005)
                this_hop = self.token_hop_len + prompt_token_pad if token_offset == 0 else self.token_hop_len
                toks = self.tts_speech_token_dict[this_uuid]
                if len(toks) - token_offset >= this_hop + PRE_LOOKAHEAD:
                    this_tok = torch.tensor(toks[:token_offset + this_hop + PRE_LOOKAHEAD]).unsqueeze(0)
                    speech = self.token2wav(this_tok, flow_prompt_speech_token, prompt_speech_feat, flow_embedding, token_offset,
                                            this_uuid, stream=True, finalize=False)
                    token_offset += this_hop
                    self.token_hop_len = min(self.token_max_hop_len, self.token_hop_len * self.stream_scale_factor)
                    yield {"tts_speech": self._to_host(speech)}
                if self.llm_end_dict[this_uuid] is True and len(self.tts_speech_token_dict[this_uuid]) - token_offset < this_hop + PRE_LOOKAHEAD:
                    break
            p.join()
            this_tok = torch.tensor(self.tts_speech_token_dict[this_uuid]).unsqueeze(0)
            speech = self.token2wav(this_tok, flow_prompt_speech_token, prompt_speech_feat, flow_embedding, token_offset, this_uuid,
                                    finalize=True)
            yield {"tts_speech": self._to_host(speech)}
        else:
            p.join()
            this_tok = torch.tensor(self.tts_speech_token_dict[this_uuid]).unsqueeze(0)
            speech = self.token2wav(this_tok, flow_prompt_speech_token, prompt_speech_feat, flow_embedding, 0, this_uuid, finalize=True,
                                    speed=speed)
            yield {"tts_speech": self._to_host(speech)}
        with self.lock:
            self.tts_speech_token_dict.pop(this_uuid)
            self.llm_end_dict.pop(this_uuid)
            self.hift_cache_dict.pop(this_uuid)
        self._release_flow_stream(this_uuid)
        self.stream.synchronize()

    # ---------------------------------------------------------------- batched streaming synthesis
    def tts_stream_batch(self, inputs, uniforms=None):
        """Streaming synthesis of several requests at once.  inputs: list of dicts with the kwargs of tts() (as for tts_batch);
        uniforms: LM sampling uniforms [steps, len(inputs), 2] (default: drawn like tts_batch).  Returns a generator of
        (i, {"tts_speech": float32 CPU [1, n]}, is_last).  Request i's chunks arrive in order and are what tts(stream=True) yields
        for it alone on a fresh model instance: same hop schedule, same mel / source / speech caches, same hamming cross-fade,
        same final non-streaming call.

        One batched LM generation runs in a thread on its own stream.  Every round collects the requests whose token count
        reached offset + hop + 3 and advances them together: ONE cvk_flow_stream_chunk_batch call on a multi-slot flow session
        for those that can use a slot, ONE prefix-recompute flow call (the reference's schedule, cli/model.py:346-363) for the
        rest (the rule of _flow_stream_chunk), then ONE vocoder call and ONE device-to-host copy for all of them.  Requests whose
        LM has ended and whose remainder is below hop + 3 finish together in one non-streaming flow call and one vocoder call.

        Differences from tts(stream=True): every request keeps its own hop (25, doubling up to token_max_hop_len), so
        self.token_hop_len - which the reference keeps on the shared instance (cli/model.py:359-360) - is neither read nor
        written.  Vocoder noise is drawn per request per chunk, in ascending request order within a round (noise_fn when set).
        Text generators (text-streaming LM) and source_speech_token (voice conversion) inputs raise ValueError."""
        for r in inputs:
            if not torch.is_tensor(r.get("text")):
                raise ValueError("tts_stream_batch: text must be a token tensor; text generators stream through tts()")
            sst = r.get("source_speech_token")
            if sst is not None and sst.shape[1] != 0:
                raise ValueError("tts_stream_batch: source_speech_token (voice conversion) streams through tts()")
        return self._stream_batch(list(inputs), uniforms)

    def _stream_batch(self, inputs, uniforms):
        B = len(inputs)
        if B == 0:
            return
        toks = [[] for _ in range(B)]
        ended = [False] * B
        taken = [{"consumed": 0, "silent": 0} for _ in range(B)]
        lm_err, lm_end = [], threading.Event()

        def progress(out_ids, out_count, live, done):
            cnt, dn, ids = out_count.tolist(), done.tolist(), out_ids.cpu()
            for b in range(B):
                self._take_tokens(ids[b], cnt[b], taken[b], toks[b])
                if dn[b]:
                    ended[b] = True                  # after its tokens: a reader that sees the flag sees every token

        def lm_job():
            try:
                self.lm_generate([r["text"] for r in inputs], [r["prompt_text"] for r in inputs], [r["llm_prompt_speech_token"] for r in inputs],
                                 uniforms, steps_per_sync=8, on_progress=progress, stream=self._new_lm_stream())
            except BaseException as e:
                lm_err.append(e)
            finally:
                lm_end.set()

        hop0 = 25                                        # cosyvoice2.yaml static chunk, the first hop of every request
        P = [int(r["flow_prompt_speech_token"].shape[1]) for r in inputs]
        pad = [int(np.ceil(p / hop0) * hop0 - p) for p in P]
        offset, hop, cache, finished = [0] * B, [hop0] * B, [None] * B, [False] * B
        # rows that may use a session slot (prompt mel 2 frames per prompt token); one slot each, sized for the longest
        slotted = [b for b in range(B) if self.incremental_flow and int(inputs[b]["prompt_speech_feat"].shape[1]) == TOKEN_MEL_RATIO * P[b]]
        cap = max([min(self.stream_cache_frames, TOKEN_MEL_RATIO * (P[b] + int(inputs[b]["text"].shape[1] * self.max_token_text_ratio)))
                   for b in slotted] + [2 * hop0])
        sess = None
        if slotted:
            try:
                sess = self._checkout_slots(len(slotted), cap)
            except cvk.CvkError:
                slotted = []                             # no memory for the caches: every request recomputes its prefixes
        slot = {b: i for i, b in enumerate(slotted)}
        lm = threading.Thread(target=lm_job, daemon=True)
        lm.start()
        try:
            while not all(finished):
                over = lm_end.is_set()
                if lm_err:
                    raise lm_err[0]
                ready, fin = [], []
                for b in range(B):
                    if finished[b]:
                        continue
                    done = ended[b] or over              # read before the token count (see progress)
                    need = hop[b] + (pad[b] if offset[b] == 0 else 0) + PRE_LOOKAHEAD
                    if len(toks[b]) - offset[b] >= need:
                        ready.append((b, toks[b][:offset[b] + need], need - PRE_LOOKAHEAD))
                    elif done:
                        fin.append(b)
                if ready:
                    mels = self._stream_round_mel(inputs, [(b, t) for b, t, _ in ready], offset, slot, sess)
                    rows = [b for b, _, _ in ready]
                    for (b, w) in zip(rows, self._stream_round_vocode(rows, mels, cache, False)):
                        yield b, {"tts_speech": w}, False
                    for b, _, this_hop in ready:
                        offset[b] += this_hop
                        hop[b] = min(self.token_max_hop_len, hop[b] * self.stream_scale_factor)
                if fin:
                    for b in fin:
                        finished[b] = True
                    rows = [b for b in fin if toks[b]]
                    outs = {}
                    if rows:
                        mel, lens = self.flow_batch([torch.tensor(toks[b], dtype=torch.int32).unsqueeze(0) for b in rows],
                                                    [inputs[b]["flow_prompt_speech_token"] for b in rows], [inputs[b]["prompt_speech_feat"] for b in rows],
                                                    [inputs[b]["flow_embedding"] for b in rows], streaming=False, finalize=True)
                        mels = [m[offset[b] * TOKEN_MEL_RATIO:] for b, m in zip(rows, torch.split(mel, lens, 0))]
                        outs = dict(zip(rows, self._stream_round_vocode(rows, mels, cache, True)))
                    for b in fin:
                        yield b, {"tts_speech": outs.get(b, torch.zeros(1, 0))}, True
                if not ready and not fin:
                    time.sleep(0.005)
        finally:
            lm.join()
            self._checkin_slots(sess)

    def _stream_round_mel(self, inputs, rows, offset, slot, sess):
        """new mel frames [n_b, 80] (device) of one round's rows (b, token prefix incl. look-ahead): ONE chunk_batch call for the
        rows that can use their session slot, ONE prefix-recompute flow call for the others.  A row that leaves the slot rule
        (chunk end off the 50-frame grid, over the slot capacity) recomputes from then on, like tts()."""
        d = self.device
        on_slot, other, new = [], [], {}
        for b, t in rows:
            P = int(inputs[b]["flow_prompt_speech_token"].shape[1])
            total = TOKEN_MEL_RATIO * (P + len(t) - PRE_LOOKAHEAD)
            done = TOKEN_MEL_RATIO * (P + offset[b]) if offset[b] else 0
            if b in slot and total % 50 == 0 and done % 50 == 0 and total <= sess[0][2]:
                on_slot.append((b, t))
            else:
                slot.pop(b, None)
                other.append((b, t))
        if on_slot:
            with torch.cuda.stream(self.stream), self.ctx.lock:
                fs = sess[1]
                for b, _ in on_slot:
                    if offset[b] == 0:
                        r = inputs[b]
                        self.ctx.flow_stream_slot_begin(fs, slot[b], r["prompt_speech_feat"][0].to(d, non_blocking=True),
                                                        r["flow_embedding"].reshape(-1).to(d, non_blocking=True))
                tl = [torch.cat([inputs[b]["flow_prompt_speech_token"].reshape(-1), torch.tensor(t, dtype=torch.int32)]).to(torch.int32)
                      for b, t in on_slot]
                mel, n = self.ctx.flow_stream_chunk_batch(fs, [slot[b] for b, _ in on_slot], tl)
                new.update(zip([b for b, _ in on_slot], torch.split(mel, n, 0)))
        if other:
            mel, lens = self.flow_batch([torch.tensor(t, dtype=torch.int32).unsqueeze(0) for _, t in other],
                                        [inputs[b]["flow_prompt_speech_token"] for b, _ in other], [inputs[b]["prompt_speech_feat"] for b, _ in other],
                                        [inputs[b]["flow_embedding"] for b, _ in other], streaming=True, finalize=False)
            for (b, _), m in zip(other, torch.split(mel, lens, 0)):
                new[b] = m[offset[b] * TOKEN_MEL_RATIO:]
        return [new[b] for b, _ in rows]

    def _stream_round_vocode(self, rows, mels, cache, finalize):
        """token2wav's vocoder half (cli/model.py:305-326) for one round's rows in ONE vocoder call (per-row cached mel frames
        and cached source) and ONE device-to-host copy; updates the rows' caches.  Returns float32 CPU [1, n] per row."""
        d = self.device
        with torch.cuda.stream(self.stream):
            tts_mels = [torch.cat([cache[b]["mel"], m], 0) if cache[b] is not None else m for b, m in zip(rows, mels)]
            lens = [int(m.shape[0]) for m in tts_mels]
            cached = [b for b in rows if cache[b] is not None]
            cs = torch.cat([cache[b]["source"] for b in cached]) if cached else None
            cl = [int(cache[b]["source"].shape[0]) if cache[b] is not None else 0 for b in rows] if cached else None
            mel = torch.cat(tts_mels, 0).contiguous()
            with self.lock:                              # one device generator shared by the request threads
                noise = torch.cat([self.noise_fn(L * SAMPLES_PER_FRAME).to(d) if self.noise_fn is not None
                                   else torch.randn(L * SAMPLES_PER_FRAME, 9, device=d, generator=self.generator) for L in lens])
        wav, src = self.hift_batch(mel, lens, cs, cl, noise=noise)
        with torch.cuda.stream(self.stream):
            outs, o = [], 0
            for b, tm, L in zip(rows, tts_mels, lens):
                w, s = wav[o:o + L * SAMPLES_PER_FRAME], src[o:o + L * SAMPLES_PER_FRAME]
                o += L * SAMPLES_PER_FRAME
                if cache[b] is not None:
                    w = self._fade_in_out(w, cache[b]["speech"])
                if not finalize:
                    cache[b] = {"mel": tm[-self.mel_cache_len:].clone(), "source": s[-self.source_cache_len:].clone(),
                                "speech": w[-self.source_cache_len:].clone()}
                    w = w[:-self.source_cache_len]
                outs.append(w)
            host = torch.cat(outs).cpu()                 # one D2H for the round
        self.stream.synchronize()
        return [c.unsqueeze(0) for c in torch.split(host, [int(w.shape[0]) for w in outs])]

    def _checkout_slots(self, n_slots, cap):
        """a multi-slot flow session ((dit, n_slots, cap), handle) with at least n_slots slots of cap frames: the idle one when it
        is large enough, else a new one (cvk.CvkError when there is no memory for it)"""
        with self._pool_lock:
            idle, self._idle_slot_session = self._idle_slot_session, None
        if idle is not None:
            (dit, n, c), fs = idle
            if dit == self.flow_stream_dit and n >= n_slots and c >= cap:
                return idle
            self.stream.synchronize()
            self.ctx.flow_stream_destroy(fs)
        with torch.cuda.stream(self.stream), self.ctx.lock:
            return (self.flow_stream_dit, n_slots, cap), self.ctx.flow_stream_slots(n_slots, cap, self.n_timesteps, dit=self.flow_stream_dit)

    def _checkin_slots(self, sess):
        """keep one idle multi-slot session for the next call; a previously idle one is destroyed"""
        if sess is None:
            return
        self.stream.synchronize()
        with self._pool_lock:
            old, self._idle_slot_session = self._idle_slot_session, sess
        if old is not None:
            self.ctx.flow_stream_destroy(old[1])
