"""CPU: batched streaming synthesis (B200CosyVoice2Model.tts_stream_batch, TtsBatcher.submit_stream) with the device primitives
faked by the oracle.  A multi-slot session's chunk returns, per slot, the frames of the streaming flow call on that slot's prefix it
has not returned yet (tests/test_flow_stream_batch_gpu.py holds the library to exactly that); the LM releases its ids a fixed number
of steps at a time, so the rounds are deterministic."""
import threading

import numpy as np
import pytest
import torch

from oracle import cases, flow, hift, lm, weights
from oracle.make_golden import stream_noise
from test_host_logic_cpu import FakeCtx2, _DummyEvent, _DummyStream, _dummy_stream_context, _pool


class FakeBatchCtx(FakeCtx2):
    """FakeCtx2 with the batched calls tts_stream_batch makes: ragged LM rows, multi-slot flow sessions, ragged flow / vocoder"""

    def __init__(self, *a):
        super().__init__(*a)
        self.batch_calls, self.hift_rows, self.flow_rows, self.destroyed = [], [], [], []
        self._memo = {}

    # ---- LM: every row decoded by the oracle with its own uniforms, released n_steps at a time
    def lm_prefill(self, sess, tt, tl, ss, sl):
        to, so = np.cumsum([0] + list(tl)), np.cumsum([0] + list(sl))
        sess.update(rows=[(tt[to[b]:to[b + 1]], ss[so[b]:so[b + 1]]) for b in range(len(tl))], ids=None, emitted=0)

    def lm_decode(self, sess, n_steps, U, min_len, max_len, out_ids, out_count, done, want_live=True):
        if sess["ids"] is None:
            sess["ids"] = []
            for b, (tt, ss) in enumerate(sess["rows"]):
                key = ("lm", tuple(tt.tolist()), tuple(ss.tolist()), U[:, b].numpy().tobytes())
                if key not in self._memo:
                    self._memo[key] = self._run(dict(tt=tt, ss=ss), U[:, b:b + 1], int(min_len[b]), int(max_len[b]))
                sess["ids"].append(self._memo[key])
        sess["emitted"] += n_steps
        live = 0
        for b, ids in enumerate(sess["ids"]):
            n = min(len(ids), sess["emitted"])
            out_ids[b, :n] = torch.tensor(ids[:n], dtype=torch.int32)
            out_count[b] = n
            done[b] = int(n == len(ids))
            live += n < len(ids)
        return live

    # ---- flow: oracle per row (memoised: rows of these tests repeat prefixes)
    def _flow(self, toks, pf, emb, streaming, finalize):
        P = self._P
        key = ("flow", tuple(toks.tolist()), pf.shape[0], pf.numpy().tobytes(), streaming, finalize)
        if key not in self._memo:
            self._memo[key] = flow.inference(self.fsd, toks[None, P:], toks[None, :P], pf[None], emb.reshape(1, -1), self.fcfg, 10,
                                             streaming, finalize)[0].t().contiguous()
        return self._memo[key]

    def flow_inference(self, toks, tl, pf, pl, emb, n_timesteps=10, streaming=False, finalize=True):
        self.flow_rows.append((len(tl), bool(streaming), bool(finalize)))
        to, po = np.cumsum([0] + list(tl)), np.cumsum([0] + list(pl))
        mels = [self._flow(toks[to[b]:to[b + 1]], pf[po[b]:po[b + 1]], emb[b], streaming, finalize) for b in range(len(tl))]
        return torch.cat(mels, 0), [m.shape[0] for m in mels]

    def flow_stream_slots(self, n_slots, max_frames, n_timesteps=10, dit=False):
        return {"slots": [None] * n_slots, "cap": max_frames}

    def flow_stream_slot_begin(self, fs, slot, prompt_feat, embedding):
        fs["slots"][slot] = {"done": 0, "pf": prompt_feat, "emb": embedding.reshape(1, -1)}

    def flow_stream_chunk_batch(self, fs, slots, tokens_list):
        assert len(set(slots)) == len(slots)
        self.batch_calls.append([int(t.numel()) for t in tokens_list])
        outs = []
        for s, toks in zip(slots, tokens_list):
            st = fs["slots"][s]
            mel = self._flow(toks, st["pf"], st["emb"], True, False)
            Tp = st["pf"].shape[0]
            outs.append(mel[max(st["done"] - Tp, 0):])
            st["done"] = Tp + mel.shape[0]
            assert st["done"] % 50 == 0 and st["done"] <= fs["cap"]
        return torch.cat(outs, 0), [o.shape[0] for o in outs]

    def flow_stream_destroy(self, fs):
        self.destroyed.append(fs)

    # ---- vocoder: ragged rows, each with its own cached source (length 0 = none yet)
    def hift_inference(self, mel, lens, noise, cache_source=None, cache_lens=None):
        self.hift_rows.append((list(lens), None if cache_lens is None else list(cache_lens)))
        wavs, srcs, o, co = [], [], 0, 0
        for b, L in enumerate(lens):
            cl = 0 if cache_lens is None else cache_lens[b]
            cs = cache_source[co:co + cl].reshape(1, 1, -1) if cl else None
            co += cl
            wav, src = hift.inference(self.hsd, mel[o:o + L].t()[None], noise[o * 480:(o + L) * 480][None], None, cs)
            wavs.append(wav[0])
            srcs.append(src.reshape(-1))
            o += L
        return torch.cat(wavs), torch.cat(srcs)


_state = {}


def _setup():
    if "ctx" not in _state:
        text, ptext, ptok, U = cases.lm_case()
        _, _, pfeat, emb = cases.flow_case(P=9)
        fcfg = flow.FlowCfg(enc_blocks=2, enc_up_blocks=1, num_mid_blocks=2, n_blocks=2)
        ctx = FakeBatchCtx(lm.synth_state_dict(2), weights.synth_state_dict(flow.param_shapes(fcfg), 1986, flow.SYNTH_GAINS),
                           weights.synth_state_dict(hift.param_shapes(), 1986, hift.SYNTH_GAINS), fcfg)
        ctx._P = ptok.shape[1]
        req = dict(text=text, flow_embedding=emb, llm_embedding=emb, prompt_text=ptext, llm_prompt_speech_token=ptok,
                   flow_prompt_speech_token=ptok, prompt_speech_feat=pfeat[:, :18])
        _state.update(ctx=ctx, req=req, U=U, pfeat=pfeat)
    return _state["ctx"], _state["req"], _state["U"]


def _model(ctx, noise_fn):
    from cosyvoice_b200.model import B200CosyVoice2Model
    m = object.__new__(B200CosyVoice2Model)
    m.ctx, m.stream, m.device = ctx, _DummyStream(), torch.device("cpu")
    m._lm_streams, m.lm_chains = [_DummyStream()], 1
    _pool(m)
    m._idle_slot_session = None
    m.uniforms_override, m.noise_fn, m.generator = None, noise_fn, None
    m.tts_speech_token_dict, m.llm_end_dict, m.hift_cache_dict = {}, {}, {}
    m.silent_tokens = []
    m.token_hop_len, m.token_max_hop_len, m.stream_scale_factor = 25, 100, 2
    m.mel_cache_len, m.source_cache_len = 8, 8 * 480
    m._window = torch.from_numpy(np.hamming(2 * 8 * 480)).float()
    m.min_token_text_ratio, m.max_token_text_ratio, m.n_timesteps = 2.0, 20.0, 10
    m.incremental_flow, m.stream_cache_frames = True, 2048
    m._new_lm_stream = lambda: _DummyStream()
    return m


def _lockstep_noise(rows):
    """noise of the k-th vocoder call of a request when `rows` requests share every round (draws in ascending request order)"""
    st = {"c": 0}

    def noise_fn(n):
        z = stream_noise(st["c"] // rows, n)
        st["c"] += 1
        return z
    return noise_fn


def _collect(gen, B):
    chunks, lasts, order = [[] for _ in range(B)], [0] * B, []
    for i, out, last in gen:
        assert not lasts[i], "a chunk after the request's last one"
        chunks[i].append(out["tts_speech"])
        lasts[i] += last
        order.append(i)
    assert lasts == [1] * B
    return chunks, order


def _check_golden(chunks, g):
    assert all(c.dtype == torch.float32 and c.shape[0] == 1 for c in chunks)
    assert [c.shape[1] for c in chunks] == g["stream_lens"].tolist()
    d = np.abs(torch.cat(chunks, 1).numpy() - g["stream_wav"])
    assert d[:, :24000].max() < 5e-3 and d.max() < 2e-2, (d[:, :24000].max(), d.max())


@pytest.fixture
def patched(monkeypatch):
    monkeypatch.setattr(torch.cuda, "Event", _DummyEvent)
    monkeypatch.setattr(torch.cuda, "stream", _dummy_stream_context)


def test_two_identical_requests_share_every_call_and_match_reference(golden, patched):
    g = golden("stream_tts")
    ctx, req, U = _setup()
    m = _model(ctx, _lockstep_noise(2))
    m.token_hop_len = 77                                 # tts_stream_batch neither reads nor writes the shared hop
    ctx.batch_calls.clear(), ctx.hift_rows.clear(), ctx.flow_rows.clear()
    chunks, order = _collect(m.tts_stream_batch([req, req], uniforms=torch.stack([U, U], 1)), 2)
    for c in chunks:
        _check_golden(c, g)
    assert order == [0, 1, 0, 1, 0, 1]                    # rounds of both rows, ascending request order inside a round
    # two streaming rounds: ONE chunk_batch call each with both rows (hop 25 padded to 41, then 50; 3 look-ahead tokens)
    assert ctx.batch_calls == [[9 + 41 + 3] * 2, [9 + 41 + 50 + 3] * 2]
    # the final, non-streaming flow call of both rows is one call; no prefix recompute
    assert ctx.flow_rows == [(2, False, True)]
    # ONE vocoder call per round, rows side by side; cached source of 3840 samples from the second call on
    assert [cl for _, cl in ctx.hift_rows] == [None, [3840, 3840], [3840, 3840]]
    assert m.token_hop_len == 77
    assert m._idle_slot_session is not None and m._idle_slot_session[0][1] == 2 and not ctx.destroyed


def test_row_off_the_slot_rule_recomputes_its_prefix(golden, patched):
    """prompt mel not 2 frames per prompt token: that row goes through the batched prefix recompute, the other keeps its slot, and
    the recomputed row's chunks equal tts(stream=True) for it alone"""
    g = golden("stream_tts")
    ctx, req, U = _setup()
    odd = dict(req, prompt_speech_feat=_state["pfeat"][:, :17])
    m = _model(ctx, _lockstep_noise(1))
    m.token_hop_len = 25
    m.uniforms_override = U[:, None, :]
    alone = [o["tts_speech"] for o in m.tts(**odd, stream=True)]
    m.uniforms_override = None
    m.noise_fn = _lockstep_noise(2)
    ctx.batch_calls.clear(), ctx.hift_rows.clear(), ctx.flow_rows.clear()
    chunks, _ = _collect(m.tts_stream_batch([req, odd], uniforms=torch.stack([U, U], 1)), 2)
    _check_golden(chunks[0], g)
    assert [c.shape[1] for c in chunks[1]] == [c.shape[1] for c in alone]
    assert np.abs(torch.cat(chunks[1], 1).numpy() - torch.cat(alone, 1).numpy()).max() < 1e-5
    assert ctx.batch_calls == [[9 + 41 + 3], [9 + 41 + 50 + 3]]                  # only row 0 on a slot
    assert ctx.flow_rows == [(1, True, False), (1, True, False), (2, False, True)]
    assert [len(lens) for lens, _ in ctx.hift_rows] == [2, 2, 2]


def test_refusals_and_empty_rows(patched):
    ctx, req, U = _setup()
    m = _model(ctx, None)
    with pytest.raises(ValueError):
        m.tts_stream_batch([dict(req, text=iter([req["text"]]))])
    with pytest.raises(ValueError):
        m.tts_stream_batch([dict(req, source_speech_token=torch.ones(1, 4, dtype=torch.int32))])
    from cosyvoice_b200.model3 import B200CosyVoice3Model
    m3 = object.__new__(B200CosyVoice3Model)
    with pytest.raises(NotImplementedError):
        m3.tts_stream_batch([req])
    assert list(m.tts_stream_batch([])) == []


# ------------------------------------------------------------------------------------------------ TtsBatcher.submit_stream
class FakeStreamModel:
    """tts_stream_batch yields, for request i, `3` chunks of 10 samples valued tag/100 + k/1000, rows interleaved"""

    def __init__(self, fail_on=None):
        self.stream_calls, self.batch_calls, self.fail_on = [], [], fail_on
        self.gate = threading.Event()

    def tts_batch(self, inputs):
        self.batch_calls.append([i["tag"] for i in inputs])
        return [torch.full((1, 10), i["tag"] / 100.0) for i in inputs]

    def tts_stream_batch(self, inputs):
        self.gate.wait()
        self.stream_calls.append([i["tag"] for i in inputs])
        for k in range(3):
            for i, r in enumerate(inputs):
                if self.fail_on == r["tag"] and k == 1:
                    raise RuntimeError("boom")
                yield i, {"tts_speech": torch.full((1, 10), r["tag"] / 100.0 + k / 1000.0)}, k == 2


def _req(tag):
    return dict(text=torch.zeros(1, 3, dtype=torch.int32), tag=tag)


def test_submit_stream_serves_a_batch_in_order():
    from cosyvoice_b200.batcher import TtsBatcher, pcm16
    m = FakeStreamModel()
    with TtsBatcher(m, max_batch=3, max_wait_ms=5000) as q:
        a, b, c = q.submit_stream(**_req(1)), q.submit_stream_pcm(**_req(2)), q.submit(**_req(3))
        m.gate.set()
        ca, cb = list(a), list(b)
        assert c.result(timeout=30).shape == (1, 10)
    assert m.stream_calls == [[1, 2]] and m.batch_calls == [[3]] and q.batches == [3]
    assert [float(x[0, 0]) for x in ca] == pytest.approx([0.01, 0.011, 0.012])
    assert cb == [pcm16(torch.full((1, 10), 0.02 + k / 1000.0)) for k in range(3)]


def test_submit_stream_failure_stays_in_its_batch():
    from cosyvoice_b200.batcher import TtsBatcher
    m = FakeStreamModel(fail_on=2)
    with TtsBatcher(m, max_batch=2, max_wait_ms=5000) as q:
        a, b = q.submit_stream(**_req(1)), q.submit_stream(**_req(2))
        m.gate.set()
        got = [next(a), next(b)]
        with pytest.raises(RuntimeError):
            list(a)
        with pytest.raises(RuntimeError):
            list(b)
        c = q.submit_stream(**_req(4))                  # the next batch is served normally
        assert len(list(c)) == 3
    assert len(got) == 2 and m.stream_calls == [[1, 2], [4]]
