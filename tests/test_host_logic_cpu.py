"""CPU: host-side control flow of the product with the device primitives replaced by oracle arithmetic.

The text-streaming LM (llm.py:551-661) is mostly control flow (5:15 interleaving, fill-token forcing, replay quirk); the
product implements it in Python over four C-ABI primitives.  Here those primitives are faked with the CPU oracle, so the
host logic of `B200CosyVoice2Model.lm_generate_bistream` is checked against the reference's golden ids without a GPU.
(The same method over the real library is checked by tests/test_lm_gpu.py::test_bistream_ids_match_reference_fp32.)"""
import contextlib
import threading

import numpy as np
import pytest
import torch

from oracle import cases, lm, sampling


def _pool(m):
    """session-pool attributes B200CosyVoice2Model.__init__ creates"""
    m._free_sessions, m._session_lru, m.max_idle_sessions, m._pool_lock = {}, [], 4, threading.Lock()
    m.flow_stream_dict, m._idle_flow_streams = {}, []
    if not hasattr(m, "lock"):
        m.lock = threading.Lock()
    return m


class FakeLmContext:
    """cvk_lm_begin / cvk_lm_feed / cvk_lm_next_logp / cvk_ras_sample semantics on oracle.lm.qwen2_forward"""

    def __init__(self, sd, num_layers):
        self.sd, self.nl = sd, num_layers
        self.lock = threading.Lock()
        self.past, self.hidden = None, None
        self.fed = []

    def lm_session(self, B, ctx_len):
        return object()

    def lm_session_destroy(self, sess):
        pass

    def lm_begin(self, sess, B=1):
        self.past, self.hidden = None, None

    def lm_feed(self, sess, ids, kinds):
        emb = []
        for i, k in zip(ids, kinds):
            table = {0: "llm.model.model.embed_tokens.weight", 1: "speech_embedding.weight", 2: "llm_embedding.weight"}[k]
            emb.append(self.sd[table][i])
        self.fed.append(len(ids))
        y, self.past = lm.qwen2_forward(self.sd, torch.stack(emb)[None], self.past, self.nl)
        self.hidden = y[:, -1]

    def lm_next_logp(self, sess, B=1):
        return lm.logprobs(self.sd, self.hidden)

    def ras_sample(self, logp, history, hist_count, uniforms, ignore_eos):
        hist = history[0, :int(hist_count[0])].tolist()
        top = sampling.ras_sample(logp[0].numpy(), hist, float(uniforms[0, 0]), float(uniforms[0, 1]), ignore_eos=bool(ignore_eos[0]))
        return torch.tensor([top], dtype=torch.int32)


def _model_with(ctx):
    from cosyvoice_b200.model import B200CosyVoice2Model
    m = object.__new__(B200CosyVoice2Model)          # no device: only the attributes the host logic touches
    m.ctx, m.stream, m.device = ctx, None, torch.device("cpu")
    m.uniforms_override, m.generator = None, None
    m.silent_tokens = []
    return _pool(m)


def test_bistream_host_logic_matches_reference(golden):
    g = golden("lm_bistream_l2")
    chunks, ptext, ptok, U = cases.bistream_case()
    ctx = FakeLmContext(lm.bistream_state_dict(2), 2)
    m = _model_with(ctx)
    ids = list(m.lm_generate_bistream(iter(chunks), ptext, ptok, uniforms=U))
    assert ids == g["ids"].tolist()
    # first model call: sos + (5 text, 15 speech) + (5 text, the 7 remaining prompt speech tokens)
    assert ctx.fed[0] == 1 + (5 + 15) + (5 + 7)
    # three calls push 5 positions: the two 5-text refills after a fill token, and the final phase, which replays the last
    # input (1 stale token embedding, llm.py:634-637) + the 3 leftover text ids + task_id (llm.py:643)
    assert ctx.fed.count(5) == 3
    assert all(n in (1, 5, 33) for n in ctx.fed)


class FakeLm3Context(FakeLmContext):
    """the same primitives for a CosyVoice3LM state_dict: llm_embedding rows 0 / 1 of the C ABI are rows 6561 / 6563 of
    speech_embedding (csrc/llm.cu llm_build), the head has no bias"""

    def lm_feed(self, sess, ids, kinds):
        emb = []
        for i, k in zip(ids, kinds):
            if k == 2:
                emb.append(self.sd["speech_embedding.weight"][(6561, 6563)[i]])
            else:
                emb.append(self.sd[{0: "llm.model.model.embed_tokens.weight", 1: "speech_embedding.weight"}[k]][i])
        self.fed.append(len(ids))
        y, self.past = lm.qwen2_forward(self.sd, torch.stack(emb)[None], self.past, self.nl)
        self.hidden = y[:, -1]

    def lm_next_logp(self, sess, B=1):
        return torch.log_softmax(torch.nn.functional.linear(self.hidden, self.sd["llm_decoder.weight"]), -1)


def test_bistream3_host_logic_matches_reference(golden):
    """CosyVoice3LM text-streaming constants (llm.py:681-684: fill 6564, eos 6562) and the <|endofprompt|> split (llm.py:583-588)
    in B200CosyVoice3Model.lm_generate_bistream: ids identical to the reference CosyVoice3LM.inference_bistream."""
    from cosyvoice_b200.model3 import B200CosyVoice3Model
    g = golden("lm3_bistream_l2")
    chunks, ptext, ptok, U = cases.bistream3_case()
    ctx = FakeLm3Context(lm.bistream_state_dict3(2), 2)
    m = object.__new__(B200CosyVoice3Model)
    m.ctx, m.stream, m.device = ctx, None, torch.device("cpu")
    m.uniforms_override, m.generator = None, None
    _pool(m)
    ids = list(m.lm_generate_bistream(iter(chunks), ptext, ptok, uniforms=U))
    assert ids == g["ids"].tolist() and int(g["trace"][-1]) == 6562
    # first model call: sos + the 3 prompt-text ids up to <|endofprompt|> + (5 text, 15 speech) + (5 text, 7 speech)
    assert ctx.fed[0] == 1 + 3 + (5 + 15) + (5 + 7)
    # without <|endofprompt|> the reference asserts (llm.py:585)
    try:
        list(m.lm_generate_bistream(iter(chunks), ptext.clamp(max=151645), ptok, uniforms=U))
        raise RuntimeError("no assertion")
    except AssertionError:
        pass


def test_llm_job_generator_branch_collects_tokens(golden):
    """cli/model.py:113-128: generator text -> bi-stream decode -> tokens appended to the session list, end flag set"""
    g = golden("lm_bistream_l2")
    chunks, ptext, ptok, U = cases.bistream_case()
    m = _model_with(FakeLmContext(lm.bistream_state_dict(2), 2))
    m.uniforms_override = U[:, None, :]
    m.tts_speech_token_dict, m.llm_end_dict = {"u": []}, {"u": False}
    m.llm_job(iter(chunks), ptext, ptok, torch.zeros(0, 192), "u")
    assert m.tts_speech_token_dict["u"] == g["ids"].tolist() and m.llm_end_dict["u"] is True


# ------------------------------------------------------------------------------------------------ CosyVoice3Model glue
class _DummyStream:
    def synchronize(self):
        pass

    def wait_event(self, e):
        pass

    def wait_stream(self, s):
        pass


class _DummyEvent:
    def __init__(self, *a, **k):
        pass

    def record(self, *a):
        pass


def _dummy_stream_context(stream):
    """torch.cuda.stream is a no-op only while no CUDA device is present; with one it would switch to the dummy stream"""
    return contextlib.nullcontext()


class FakeCtx3:
    """the libcvk calls B200CosyVoice3Model makes (batched LM session API, flow3, hift3) on the CPU oracles"""

    def __init__(self, lsd, fsd, hsd, depth, rand_ini, sine_noise):
        from oracle import dit, hift_causal
        self.lsd, self.fsd, self.hsd, self.depth = lsd, fsd, hsd, depth
        self.rand_ini, self.sine_noise = rand_ini, sine_noise
        self.dit, self.hc = dit, hift_causal
        self.lock = threading.Lock()
        self.flow_calls, self.hift_calls, self.stream_calls = [], [], []

    # ---- cvk_flow_stream_* / cvk_flow3_stream_create: a session returns, per chunk, the frames of the streaming flow call on the prefix
    # that it has not returned yet (tests/test_flow_gpu.py / test_flow3_gpu.py hold the library to exactly that)
    def flow_stream(self, max_frames, n_timesteps=10, dit=False):
        return {"done": 0, "cap": max_frames, "dit": dit}

    def flow_stream_begin(self, fs, prompt_feat, embedding):
        fs.update(done=0, pf=prompt_feat, emb=embedding.reshape(1, -1))

    def _prefix_mel(self, fs, toks):
        assert fs["dit"]
        P = self._P
        return self.dit.inference(self.fsd, toks[None, P:], toks[None, :P], fs["pf"][None], fs["emb"], self.depth, 10, True, False)[0].t()

    def flow_stream_chunk(self, fs, toks):
        self.stream_calls.append(int(toks.numel()))
        mel = self._prefix_mel(fs, toks)
        Tp = fs["pf"].shape[0]
        out = mel[max(fs["done"] - Tp, 0):]
        fs["done"] = Tp + mel.shape[0]
        assert fs["done"] % 50 == 0 and fs["done"] <= fs["cap"]
        return out.contiguous()

    def flow_stream_destroy(self, fs):
        pass

    # ---- LM: prefill stores the prompt, decode releases the oracle's ids n_steps at a time
    def lm_session(self, B, ctx_len):
        return {"ids": None, "emitted": 0}

    def lm_session_destroy(self, sess):
        pass

    def lm_prefill(self, sess, tt, tl, ss, sl):
        sess.update(tt=tt.clone(), ss=ss.clone(), ids=None, emitted=0)

    def _run(self, sess, U, min_len, max_len):
        sd = self.lsd
        emb = torch.nn.functional.embedding
        lm_in = torch.cat([sd["speech_embedding.weight"][6561].reshape(1, 1, -1), emb(sess["tt"].long()[None], sd["llm.model.model.embed_tokens.weight"]),
                           sd["speech_embedding.weight"][6563].reshape(1, 1, -1), emb(sess["ss"].long()[None], sd["speech_embedding.weight"])], 1)
        out, past = [], None
        for i in range(max_len):
            y, past = lm.qwen2_forward(sd, lm_in, past, 2)
            logp = torch.log_softmax(torch.nn.functional.linear(y[:, -1], sd["llm_decoder.weight"]), -1)[0]
            top = sampling.ras_sample(logp.numpy(), out, float(U[i, 0, 0]), float(U[i, 0, 1]), ignore_eos=i < min_len)
            if top >= 6561:
                break
            out.append(top)
            lm_in = sd["speech_embedding.weight"][top].reshape(1, 1, -1)
        return out

    def lm_decode(self, sess, n_steps, U, min_len, max_len, out_ids, out_count, done, want_live=True):
        if sess["ids"] is None:
            sess["ids"] = self._run(sess, U, int(min_len[0]), int(max_len[0]))
        ids = sess["ids"]
        sess["emitted"] = min(len(ids), sess["emitted"] + n_steps)
        n = sess["emitted"]
        out_ids[0, :n] = torch.tensor(ids[:n], dtype=torch.int32)
        out_count[0] = n
        finished = n == len(ids)
        done[0] = int(finished)
        return 0 if finished else 1

    # ---- flow / vocoder
    def flow3_inference(self, toks, tl, pf, pl, emb, n_timesteps=10, streaming=False, finalize=True):
        P = self._P
        self.flow_calls.append((int(tl[0]), bool(streaming), bool(finalize)))
        mel = self.dit.inference(self.fsd, toks[None, P:], toks[None, :P], pf[None], emb, self.depth, n_timesteps, streaming, finalize)
        return mel[0].t().contiguous(), [mel.shape[2]]

    def hift3_inference(self, mel, lens, finalize=True):
        self.hift_calls.append((int(lens[0]), bool(finalize)))
        wav, src = self.hc.inference(self.hsd, mel.t()[None], self.rand_ini, self.sine_noise, finalize)
        return wav[0], None, src.reshape(-1)


def test_cosyvoice3_model_host_glue_matches_reference(golden, monkeypatch):
    """B200CosyVoice3Model.tts / token2wav / llm_job (cli/model.py:397-450 + inherited :328-394) with the device primitives faked by
    the oracle: the chunk schedule, the growing mel cache and the speech_offset bookkeeping reproduce the reference's own
    CosyVoice3Model.tts (tests/golden/stream3_tts.npz), offline and streaming."""
    from cosyvoice_b200.model3 import B200CosyVoice3Model
    from oracle import dit, hift_causal as hc, weights
    monkeypatch.setattr(torch.cuda, "Event", _DummyEvent)
    monkeypatch.setattr(torch.cuda, "stream", _dummy_stream_context)
    g = golden("stream3_tts")
    text, ptext, ptok, U = cases.lm3_case()
    _, _, pfeat, emb = cases.flow_case(P=9)
    pfeat = pfeat[:, :18]
    _, rand_ini, sine_noise = cases.hift_causal_case(T=400)
    ctx = FakeCtx3(lm.synth_state_dict3(2), weights.synth_state_dict(dit.flow_param_shapes(2), 1986, dit.SYNTH_GAINS),
                   weights.synth_state_dict(hc.param_shapes(), 1986, hc.SYNTH_GAINS), 2, rand_ini, sine_noise)
    ctx._P = ptok.shape[1]
    for mode, stream in (("offline", False), ("stream", True)):
        m = object.__new__(B200CosyVoice3Model)
        m.ctx, m.stream, m.device = ctx, _DummyStream(), torch.device("cpu")
        m._lm_streams, m.lm_chains = [_DummyStream()], 1
        _pool(m)
        m.uniforms_override, m.noise_fn, m.generator = U[:, None, :], None, None
        m.lock = threading.Lock()
        m.tts_speech_token_dict, m.llm_end_dict, m.hift_cache_dict = {}, {}, {}
        m.silent_tokens = [1, 2, 28, 29, 55, 248, 494, 2241, 2242, 2322, 2323]
        m.token_hop_len, m.token_max_hop_len, m.stream_scale_factor = 25, 100, 2
        m.min_token_text_ratio, m.max_token_text_ratio, m.n_timesteps = 2.0, 20.0, 10
        for incremental in ((True, False) if stream else (True,)):
            m.incremental_flow = incremental
            m.token_hop_len = 25
            ctx.flow_calls.clear()
            ctx.hift_calls.clear()
            ctx.stream_calls.clear()
            chunks = [o["tts_speech"] for o in m.tts(text=text, flow_embedding=emb, llm_embedding=emb, prompt_text=ptext,
                                                     llm_prompt_speech_token=ptok, flow_prompt_speech_token=ptok, prompt_speech_feat=pfeat,
                                                     stream=stream)]
            assert [c.shape[1] for c in chunks] == g[mode + "_lens"].tolist()
            d = np.abs(torch.cat(chunks, 1).numpy() - g[mode + "_wav"])
            assert d[:, :24000].max() < 2e-3 and d.max() < 1e-2
            assert not m.flow_stream_dict
            if stream and incremental:
                # DiT sessions for the two streaming chunks, flow3_inference for the final non-streaming call
                assert ctx.stream_calls == [9 + 41 + 3, 9 + 41 + 50 + 3] and ctx.flow_calls == [(9 + 140, False, True)]
        if stream:
            # last pass = the reference's schedule: two streaming calls on growing prefixes (hop 25 padded to 41, then 50; 3 look-ahead
            # tokens each) + the final non-streaming call on all 140 tokens (cli/model.py:346-373)
            assert ctx.flow_calls == [(9 + 41 + 3, True, False), (9 + 41 + 50 + 3, True, False), (9 + 140, False, True)]
            assert [f for _, f in ctx.hift_calls] == [False, False, True]
            assert m.token_hop_len == 100


# ------------------------------------------------------------------------------------------------ CosyVoice2Model glue
class FakeCtx2(FakeCtx3):
    """libcvk calls of B200CosyVoice2Model (Qwen2LM session API, flow_inference, hift_inference with cache_source) on the oracles"""

    def __init__(self, lsd, fsd, hsd, fcfg):
        self.lsd, self.fsd, self.hsd, self.fcfg = lsd, fsd, hsd, fcfg
        self.lock = threading.Lock()
        self.flow_calls, self.hift_calls, self.stream_calls = [], [], []

    def _prefix_mel(self, fs, toks):
        from oracle import flow
        assert not fs["dit"]
        P = self._P
        return flow.inference(self.fsd, toks[None, P:], toks[None, :P], fs["pf"][None], fs["emb"], self.fcfg, 10, True, False)[0].t()

    def _run(self, sess, U, min_len, max_len):
        sd = self.lsd
        emb = torch.nn.functional.embedding
        lm_in = torch.cat([sd["llm_embedding.weight"][0].reshape(1, 1, -1), emb(sess["tt"].long()[None], sd["llm.model.model.embed_tokens.weight"]),
                           sd["llm_embedding.weight"][1].reshape(1, 1, -1), emb(sess["ss"].long()[None], sd["speech_embedding.weight"])], 1)
        out, past = [], None
        for i in range(max_len):
            y, past = lm.qwen2_forward(sd, lm_in, past, 2)
            top = sampling.ras_sample(lm.logprobs(sd, y[:, -1])[0].numpy(), out, float(U[i, 0, 0]), float(U[i, 0, 1]), ignore_eos=i < min_len)
            if top in lm.STOP_IDS:
                break
            out.append(top)
            lm_in = sd["speech_embedding.weight"][top].reshape(1, 1, -1)
        return out

    def flow_inference(self, toks, tl, pf, pl, emb, n_timesteps=10, streaming=False, finalize=True):
        from oracle import flow
        P = self._P
        self.flow_calls.append((int(tl[0]), bool(streaming), bool(finalize)))
        mel = flow.inference(self.fsd, toks[None, P:], toks[None, :P], pf[None], emb, self.fcfg, n_timesteps, streaming, finalize)
        return mel[0].t().contiguous(), [mel.shape[2]]

    def hift_inference(self, mel, lens, noise, cache_source=None, cache_lens=None):
        from oracle import hift
        self.hift_calls.append((int(lens[0]), 0 if cache_source is None else int(cache_source.numel())))
        cs = cache_source.reshape(1, 1, -1) if cache_source is not None else None
        wav, src = hift.inference(self.hsd, mel.t()[None], noise[None], None, cs)
        return wav[0], src.reshape(-1)


def test_cosyvoice2_model_host_glue_matches_reference(golden, monkeypatch):
    """B200CosyVoice2Model.tts / token2wav / llm_job (cli/model.py:245-394) with the device primitives faked by the oracle:
    chunk schedule, mel / source / speech caches and the hamming cross-fade reproduce the reference's own CosyVoice2Model.tts
    (tests/golden/stream_tts.npz), offline and streaming.  (The same class over the real library: tests/test_model_gpu.py.)"""
    from cosyvoice_b200.model import B200CosyVoice2Model
    from oracle import flow, hift, weights
    from oracle.make_golden import stream_noise
    monkeypatch.setattr(torch.cuda, "Event", _DummyEvent)
    monkeypatch.setattr(torch.cuda, "stream", _dummy_stream_context)
    g = golden("stream_tts")
    text, ptext, ptok, U = cases.lm_case()
    _, _, pfeat, emb = cases.flow_case(P=9)
    pfeat = pfeat[:, :18]
    fcfg = flow.FlowCfg(enc_blocks=2, enc_up_blocks=1, num_mid_blocks=2, n_blocks=2)
    ctx = FakeCtx2(lm.synth_state_dict(2), weights.synth_state_dict(flow.param_shapes(fcfg), 1986, flow.SYNTH_GAINS),
                   weights.synth_state_dict(hift.param_shapes(), 1986, hift.SYNTH_GAINS), fcfg)
    ctx._P = ptok.shape[1]
    for mode, stream in (("offline", False), ("stream", True)):
        k = {"k": 0}

        def noise_fn(n):
            z = stream_noise(k["k"], n)
            k["k"] += 1
            return z
        m = object.__new__(B200CosyVoice2Model)
        m.ctx, m.stream, m.device = ctx, _DummyStream(), torch.device("cpu")
        m._lm_streams, m.lm_chains = [_DummyStream()], 1
        _pool(m)
        m.uniforms_override, m.noise_fn, m.generator = U[:, None, :], noise_fn, None
        m.lock = threading.Lock()
        m.tts_speech_token_dict, m.llm_end_dict, m.hift_cache_dict = {}, {}, {}
        m.silent_tokens = []
        m.token_hop_len, m.token_max_hop_len, m.stream_scale_factor = 25, 100, 2
        m.mel_cache_len, m.source_cache_len = 8, 8 * 480
        m._window = torch.from_numpy(np.hamming(2 * 8 * 480)).float()
        m.min_token_text_ratio, m.max_token_text_ratio, m.n_timesteps = 2.0, 20.0, 10
        for incremental in ((True, False) if stream else (True,)):
            m.incremental_flow = incremental
            m.token_hop_len = 25
            k["k"] = 0
            ctx.flow_calls.clear()
            ctx.hift_calls.clear()
            ctx.stream_calls.clear()
            chunks = [o["tts_speech"] for o in m.tts(text=text, flow_embedding=emb, llm_embedding=emb, prompt_text=ptext,
                                                     llm_prompt_speech_token=ptok, flow_prompt_speech_token=ptok, prompt_speech_feat=pfeat,
                                                     stream=stream)]
            assert [c.shape[1] for c in chunks] == g[mode + "_lens"].tolist()
            d = np.abs(torch.cat(chunks, 1).numpy() - g[mode + "_wav"])
            assert d[:, :24000].max() < 5e-3 and d.max() < 2e-2, (d[:, :24000].max(), d.max())
            assert not m.flow_stream_dict                    # the session went back to the pool
            if stream and incremental:
                # the two streaming chunks (hop 25 padded to 41, then 50; 3 look-ahead tokens each) through the cached session, the
                # final non-streaming call on all 140 tokens through flow_inference like the reference (cli/model.py:372-378)
                assert ctx.stream_calls == [9 + 41 + 3, 9 + 41 + 50 + 3]
                assert ctx.flow_calls == [(9 + 140, False, True)]
        if stream:
            # last pass = the reference's schedule: prefix recompute for every chunk
            assert ctx.flow_calls == [(9 + 41 + 3, True, False), (9 + 41 + 50 + 3, True, False), (9 + 140, False, True)]
            assert ctx.stream_calls == []
            assert len(m._idle_flow_streams) == 1
            # every vocoder call after the first re-uses 8 cached mel frames and 3840 cached source samples (cli/model.py:305-318)
            assert [c[1] for c in ctx.hift_calls] == [0, 3840, 3840]


def test_padded_cosyvoice3_head_is_sampling_neutral():
    """The CosyVoice3LM stage pads the 6761-way head to 6764 outputs whose bias is -1e30 (csrc/llm.cu): after the log-softmax the
    pad ids have probability exactly 0, every real log-prob is bit-identical, and repetition-aware sampling draws the same ids."""
    g = np.random.default_rng(5)
    for temp in (0.7, 3.0, 8.0):
        logits = (g.standard_normal(6761) * temp).astype(np.float32)
        padded = np.concatenate([logits, np.full(3, -1.0e30, dtype=np.float32)])
        lp, lpp = sampling.log_softmax_f32(logits), sampling.log_softmax_f32(padded)
        assert np.array_equal(lp, lpp[:6761]) and np.all(np.exp(lpp[6761:].astype(np.float64)) == 0.0)
        hist = [int(np.argmax(logits))] * 3
        for u1, u2, ign in ((0.05, 0.9, True), (0.5, 0.5, False), (0.79, 0.01, True), (0.999, 0.999, False)):
            assert sampling.ras_sample(lp, hist, u1, u2, ign) == sampling.ras_sample(lpp, hist, u1, u2, ign)


def test_frontend_wrappers_refuse_configurations_the_library_does_not_implement():
    """cosyvoice_b200/frontend.py: argument checks happen before any device work (no silent fallback to another configuration)"""
    from cosyvoice_b200 import frontend
    w = torch.zeros(1, 16000)
    with pytest.raises(ValueError):
        frontend.kaldi_fbank(w, num_mel_bins=40)
    with pytest.raises(ValueError):
        frontend.kaldi_fbank(w, dither=1.0)
    with pytest.raises(ValueError):
        frontend.kaldi_fbank(torch.zeros(2, 16000))
    with pytest.raises(ValueError):
        frontend.log_mel_spectrogram(w, n_mels=80)
    with pytest.raises(ValueError):
        frontend.mel_spectrogram(torch.zeros(1, 24000), n_fft=1024)
    with pytest.raises(ValueError):
        frontend.mel_spectrogram(torch.zeros(1, 24000), fmax=7600)
