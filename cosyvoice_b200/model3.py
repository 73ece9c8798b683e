"""Host-side mirror of the reference's CosyVoice3Model (cosyvoice/cli/model.py:397-450) over libcvk.

CosyVoice3Model inherits CosyVoice2Model.tts (thread-per-request LM job, chunk schedule hop 25 -> 50 -> 100 with 3 look-ahead
tokens) and replaces token2wav: the flow is the DiT one (stage "flow3"), the vocoder is the causal one (stage "hift3"), and instead
of the CosyVoice2 mel / source / speech caches with a cross-fade it keeps ALL mel frames produced so far, re-runs the causal vocoder
over them and emits the samples beyond ``speech_offset``.  This class follows that bookkeeping literally.

Status (end of round 1): the flow stage is parity-green on the GPU; the LM variant and the vocoder (offline and streaming call)
are written but had their first GPU run only at the round-end test pass.  The class itself is checked on the CPU against the reference's own
CosyVoice3Model.tts with the device primitives faked by the oracle (tests/test_host_logic_cpu.py)."""
import torch

from .model import B200CosyVoice2Model, TOKEN_MEL_RATIO, _count


class B200CosyVoice3Model(B200CosyVoice2Model):
    # CosyVoice3LM (llm.py:681-684): sos 6561 / eos 6562 / task_id 6563 / fill 6564; <|endofprompt|> = 151646 (llm.py:585)
    bistream_fill_token = 6564
    bistream_eos_token = 6562
    bistream_eop_token = 151646
    flow_stream_dit = True            # streaming chunks through cvk_flow3_stream_create sessions (DiT K/V + position-convolution tails)

    def __init__(self, *a, **k):
        super().__init__(*a, **k)
        # FSQ silent and breath tokens (cli/model.py:423)
        self.silent_tokens = [1, 2, 28, 29, 55, 248, 494, 2241, 2242, 2322, 2323]

    # ---------------------------------------------------------------- weights
    def load_state_dicts(self, llm_sd, flow_sd, hift_sd, rand_ini=None, sine_noise=None):
        """llm_sd: CosyVoice3LM, flow_sd: CausalMaskedDiffWithDiT, hift_sd: CausalHiFTGenerator state_dicts.  rand_ini [1,9] /
        sine_noise [1,n,9]: the vocoder's constructor-time random tensors (SineGen2.rand_ini / .sine_waves, generator.py:223-226),
        which are module attributes and not part of the state_dict; drawn like the reference draws them when omitted."""
        from .model import cfm_rand_noise
        nl = _count(llm_sd.keys(), "llm.model.model.layers.")
        depth = _count(list(flow_sd.keys()), "decoder.estimator.transformer_blocks.")
        self.ctx.load_state_dict("llm", llm_sd, [nl])
        self.ctx.load_state_dict("flow3", flow_sd, [depth])
        self.ctx.load_state_dict("hift3", hift_sd)
        self.ctx.set_cfm_noise(cfm_rand_noise())
        if rand_ini is None:
            rand_ini = torch.rand(1, 9)
            rand_ini[:, 0] = 0
        if sine_noise is None:
            sine_noise = torch.rand(1, 300 * 24000, 9)
        self.ctx.hift3_set_noise(rand_ini, sine_noise.reshape(-1, 9))

    # ---------------------------------------------------------------- flow + vocoder
    def flow_batch(self, tokens, prompt_tokens, prompt_feats, embeddings, streaming=False, finalize=True):
        d = self.device
        tl = [int(t.shape[1] + p.shape[1]) for t, p in zip(tokens, prompt_tokens)]
        pl = [int(f.shape[1]) for f in prompt_feats]
        with torch.cuda.stream(self.stream), self.ctx.lock:
            toks = torch.cat([torch.cat([p.reshape(-1).to(d), t.reshape(-1).to(d)]) for t, p in zip(tokens, prompt_tokens)]).to(torch.int32)
            pf = torch.cat([f[0].to(d) for f in prompt_feats], 0) if sum(pl) else None
            emb = torch.cat([e.reshape(1, -1).to(d) for e in embeddings], 0)
            return self.ctx.flow3_inference(toks, tl, pf, pl, emb, n_timesteps=self.n_timesteps, streaming=streaming, finalize=finalize)

    def token2wav(self, token, prompt_token, prompt_feat, embedding, token_offset, uuid, stream=False, finalize=False, speed=1.0):
        """cli/model.py:425-450"""
        new_mel = self._flow_stream_chunk(token.to(torch.int32), prompt_token, prompt_feat, embedding, token_offset, uuid) \
            if (stream and not finalize) else None
        if new_mel is None:
            mel, _ = self.flow_batch([token.to(torch.int32)], [prompt_token], [prompt_feat], [embedding], streaming=stream, finalize=finalize)
        with torch.cuda.stream(self.stream):
            tts_mel = new_mel if new_mel is not None else mel[token_offset * TOKEN_MEL_RATIO:]
            cache = self.hift_cache_dict[uuid]
            if cache is not None:
                tts_mel = torch.cat([cache["mel"], tts_mel], 0)
                cache["mel"] = tts_mel
            else:
                cache = self.hift_cache_dict[uuid] = {"mel": tts_mel, "speech_offset": 0}
            if speed != 1.0:
                assert token_offset == 0 and finalize is True, "speed change only support non-stream inference mode"
                m = torch.nn.functional.interpolate(tts_mel.t().unsqueeze(0), size=int(tts_mel.shape[0] / speed), mode="linear")
                tts_mel = m[0].t()
            with self.ctx.lock:
                wav, _, _ = self.ctx.hift3_inference(tts_mel.contiguous(), [tts_mel.shape[0]], finalize=finalize)
            wav = wav[cache["speech_offset"]:]
            cache["speech_offset"] += wav.shape[0]
        return wav.unsqueeze(0)

    def tts_stream_batch(self, inputs, uniforms=None):
        """Not available for CosyVoice3: its token2wav keeps every mel frame and re-runs the causal vocoder over them, a different
        schedule from the CosyVoice2 caches that B200CosyVoice2Model.tts_stream_batch batches.  Stream through tts()."""
        raise NotImplementedError("tts_stream_batch is CosyVoice2 only; CosyVoice3 streams through tts(stream=True)")
