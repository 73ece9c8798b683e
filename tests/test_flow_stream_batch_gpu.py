"""GPU: batched streaming synthesis.  Multi-slot streaming-flow sessions (cvk_flow_stream_slots_create / _slot_begin /
_chunk_batch) against one-slot sessions and against the reference's prefix recompute (flow.inference(streaming=True,
finalize=False) on the growing prefix, cli/model.py:346-363); B200CosyVoice2Model.tts_stream_batch against the reference's own
CosyVoice2Model.tts (tests/golden/stream_tts.npz) and against tts(stream=True); TtsBatcher.submit_stream over the real model."""
import pytest
import torch

from gpu_util import maxdiff
from oracle.make_golden import stream_noise
from test_flow3_gpu import model as dit_model
from test_flow_gpu import model as unet_model
from test_model_gpu import model as tts_model, request

pytestmark = pytest.mark.gpu


def _slot_case(seed):
    """3 utterances: prompts of 30 / 9 / 0 tokens, own embeddings, own tokens; hop schedules of tts() (first hop padded to the
    25-token grid, then doubling).  10 spare tokens past the last look-ahead feed the off-grid refusal."""
    g = torch.Generator().manual_seed(seed)
    utts = []
    for P, hops in ((30, (45, 25, 50)), (9, (41, 50)), (0, (25, 50))):
        utts.append(dict(P=P, hops=hops, toks=torch.randint(0, 6561, (P + sum(hops) + 3 + 10,), generator=g, dtype=torch.int32),
                         pfeat=torch.rand(2 * P, 80, generator=g) * 13.5 - 11.5, emb=torch.randn(1, 192, generator=g)))
    return utts


@pytest.mark.parametrize("kind,precision,tag", [
    ("unet", "fp32", "small"), ("unet", "bf16", "small"), ("unet", "bf16", "full"), ("dit", "fp32", 2), ("dit", "bf16", 2)])
def test_chunk_batch_equals_one_slot_sessions_and_prefix_recompute(kind, precision, tag):
    """Slots at different chunk positions, with different prompt lengths and chunk lengths, advance in one call: every slot's
    frames equal a one-slot session fed the same prefixes and the reference schedule's prefix recompute.  Slot 0 is on its third
    chunk while slot 2 is on its first, passed in the order [2, 0].  Refused calls (duplicate slot, slot not begun, chunk end off
    the 50-frame grid, slot out of range) raise and modify nothing: the next valid call still matches."""
    from cosyvoice_b200.cvk import CvkError
    dit = kind == "dit"
    c = dit_model(precision, tag) if dit else unet_model(precision, tag)[0]
    recompute = c.flow3_inference if dit else c.flow_inference
    tol = 1e-5 if precision == "fp32" else 1e-3
    utts = _slot_case(91)
    # expected frames per (slot, chunk): prefix recompute, and a one-slot session per utterance
    want, one = {}, {}
    for s, u in enumerate(utts):
        fs1 = c.flow_stream(max_frames=512, n_timesteps=10, dit=dit)
        try:
            c.flow_stream_begin(fs1, u["pfeat"], u["emb"])
            n, done = u["P"], 0
            for k, hop in enumerate(u["hops"]):
                n += hop
                ref, _ = recompute(u["toks"][:n + 3], [n + 3], u["pfeat"], [2 * u["P"]], u["emb"], streaming=True, finalize=False)
                want[s, k] = ref[max(done - 2 * u["P"], 0):]
                one[s, k] = c.flow_stream_chunk(fs1, u["toks"][:n + 3])
                done = 2 * n
        finally:
            c.flow_stream_destroy(fs1)
    fs = c.flow_stream_slots(4, max_frames=512, n_timesteps=10, dit=dit)       # slot 3 is never begun
    pos = [0, 0, 0]                                                              # chunks delivered per slot
    worst = [0.0]

    def prefix(s, extra=0):
        u = utts[s]
        return u["toks"][:u["P"] + sum(u["hops"][:pos[s] + 1]) + extra + 3]

    def step(slots):
        mel, n = c.flow_stream_chunk_batch(fs, slots, [prefix(s) for s in slots])
        for s, m in zip(slots, torch.split(mel, n, 0)):
            w = want[s, pos[s]]
            assert m.shape == w.shape, (s, pos[s], m.shape, w.shape)
            assert torch.isfinite(m).all()
            d = max(maxdiff(m, w), maxdiff(m, one[s, pos[s]]))
            worst[0] = max(worst[0], d)
            assert d < tol, (s, pos[s], d)
            pos[s] += 1
    try:
        assert c.flow_stream_bytes(fs) > 0
        for s, u in enumerate(utts):
            c.flow_stream_slot_begin(fs, s, u["pfeat"], u["emb"])
        step([0])
        step([0, 1])
        for bad_slots, bad_toks in (([0, 0], [prefix(0), prefix(0)]), ([3], [prefix(0)]), ([1], [prefix(1, extra=10)]),
                                    ([7], [prefix(0)]), ([2, 1], [prefix(2), prefix(1, extra=10)])):
            with pytest.raises(CvkError):
                c.flow_stream_chunk_batch(fs, bad_slots, bad_toks)
        step([2, 0])
        step([1, 2])
        assert pos == [3, 2, 2]
        print(f"[{kind} {precision} {tag}] max |chunk_batch - reference| = {worst[0]:.3g}")
    finally:
        c.flow_stream_destroy(fs)


# ------------------------------------------------------------------------------------------------ model level
def _noise_by_length(m, req, U):
    """vocoder noise as a function of the sample count only, so that a row's audio does not depend on which rows share its
    rounds: the k-th vocoder call of tts(stream=True) for `req` (the golden's schedule) gets stream_noise(k, n)"""
    sizes = []

    def rec(n):
        sizes.append(n)
        return stream_noise(len(sizes) - 1, n).to(m.device)
    m.uniforms_override, m.noise_fn, m.token_hop_len = U[:, None, :], rec, 25
    list(m.tts(**req, stream=True))
    k_of = {n: k for k, n in enumerate(sizes)}
    assert len(k_of) == len(sizes)
    m.uniforms_override, m.noise_fn = None, None
    return lambda n: stream_noise(k_of.get(n, 1000 + n), n).to(m.device)


def _check_golden(chunks, g):
    assert [c.shape[1] for c in chunks] == g["stream_lens"].tolist()
    assert all(c.device.type == "cpu" and c.dtype == torch.float32 and c.shape[0] == 1 for c in chunks)
    _check_close(torch.cat(chunks, 1), torch.from_numpy(g["stream_wav"]))


def _check_close(wav, ref):
    # bounds of tests/test_model_gpu.py::test_tts_matches_reference_model
    d_head = maxdiff(wav[:, :24000], ref[:, :24000])
    rel = ((wav - ref).norm() / ref.norm()).item()
    assert d_head < 5e-3, d_head
    assert rel < 0.05, rel


def _collect(gen, B):
    chunks, lasts = [[] for _ in range(B)], [0] * B
    for i, out, last in gen:
        assert not lasts[i]
        chunks[i].append(out["tts_speech"])
        lasts[i] += last
    assert lasts == [1] * B
    return chunks


def test_tts_stream_batch_reproduces_reference_and_single_requests(golden):
    g = golden("stream_tts")
    m = tts_model()
    req, U = request()
    noise = _noise_by_length(m, req, U)
    m.token_hop_len = 25
    try:
        m.noise_fn = noise
        (alone,) = _collect(m.tts_stream_batch([req], uniforms=U[:, None, :]), 1)
        _check_golden(alone, g)
        # two copies of the request and a different one, per-row uniforms
        req2 = dict(req)
        g2 = torch.Generator().manual_seed(123)
        req2["text"] = torch.randint(0, 151643, (1, 5), generator=g2, dtype=torch.int32)
        Ub = torch.rand(U.shape[0], 3, 2, generator=g2)
        Ub[:, 0] = U
        Ub[:, 1] = U
        m.token_hop_len = 33                          # neither read nor written by tts_stream_batch
        rows = _collect(m.tts_stream_batch([req, req, req2], uniforms=Ub), 3)
        assert m.token_hop_len == 33
        assert [c.shape for c in rows[0]] == [c.shape for c in rows[1]]
        assert all(torch.equal(a, b) for a, b in zip(rows[0], rows[1]))
        _check_golden(rows[0], g)
        # row 2 against tts(stream=True) for req2 alone on a fresh hop
        m.token_hop_len = 25
        m.uniforms_override = Ub[:, 2:3, :].contiguous()
        ref2 = [o["tts_speech"] for o in m.tts(**req2, stream=True)]
        assert [c.shape[1] for c in rows[2]] == [c.shape[1] for c in ref2]
        _check_close(torch.cat(rows[2], 1), torch.cat(ref2, 1))
        assert m._idle_slot_session is not None
    finally:
        m.uniforms_override, m.noise_fn = None, None


def test_batcher_serves_two_streams_as_one_batch(golden):
    from cosyvoice_b200.batcher import TtsBatcher
    g = golden("stream_tts")
    m = tts_model()
    req, U = request()
    noise = _noise_by_length(m, req, U)
    try:
        m.noise_fn = noise
        m.uniforms_override = U[:, None, :].expand(-1, 2, -1).contiguous()
        with TtsBatcher(m, max_batch=2, max_wait_ms=5000) as q:
            a, b = q.submit_stream(**req), q.submit_stream(**req)
            ca, cb = list(a), list(b)
        assert q.batches == [2]
        _check_golden(ca, g)
        _check_golden(cb, g)
    finally:
        m.uniforms_override, m.noise_fn = None, None
