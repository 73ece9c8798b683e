"""GPU: parity of the BENCHMARKED mode (bf16 tensor-core operands, persistent LM decode kernel) at the BENCHMARK shape - one
full-size Z10 utterance (24-layer LM over 389 positions, 325 tokens -> 650 mel frames through the full flow, 500 frames through the
vocoder) against the CPU oracle's outputs committed in tests/golden/z10_full.npz (oracle/make_golden_full.py; the vocoder's source
and waveform are recomputed from the committed mel and checked against committed samples).

SURVEY.md §8(c)(iii) protocol: teacher-forced log-probs (max |d| and top-25 set overlap), mel after 10 Euler steps against fp32 with
the reference-style 16-bit autocast deviation printed beside it as the yardstick, waveform with the source injected.  Every test
prints the MEASURED deviation; the asserted bounds are those measurements with head-room, not aspirations."""
import numpy as np
import pytest
import torch

from gpu_util import maxdiff
from oracle import flow, hift, lm, weights
from oracle.make_golden_full import LM_ROWS, PIN_STRIDE, case

pytestmark = pytest.mark.gpu
_c = {}


def bctx():
    from cosyvoice_b200 import cvk
    if "c" not in _c:
        _c["c"] = cvk.Context(0, "bf16", workspace_gb=8.0)
    return _c["c"]


def test_lm_teacher_forced_logp_fullsize(golden):
    g = golden("z10_full")
    c = bctx()
    sd = lm.synth_state_dict(24)
    c.load_state_dict("llm", sd, cfg=[24])
    utt, ids, _ = case()
    lm_in = lm.build_lm_input(sd, utt["text"], utt["prompt_text"], utt["llm_prompt_speech_token"])
    full = torch.cat([lm_in, torch.nn.functional.embedding(ids[None], sd["speech_embedding.weight"])], 1)[0]
    logp = c.lm_forward_logp(full, [full.shape[0]]).cpu()
    L0 = lm_in.shape[1]
    got = logp[[L0 - 1 + r for r in LM_ROWS]]
    ref = torch.from_numpy(g["lm_logp"])
    d = (got - ref).abs().max().item()
    overlap = []
    for i in range(ref.shape[0]):
        a, b = set(ref[i].topk(25).indices.tolist()), set(got[i].topk(25).indices.tolist())
        overlap.append(len(a & b))
    am = int((got.argmax(-1) == ref.argmax(-1)).sum())
    print(f"[full-size LM, bf16] max |dlogp| {d:.4g} on |logp| <= {ref.abs().max().item():.3g}; top-25 overlap per row {overlap}; arg-max equal {am}/{ref.shape[0]}")
    assert d < 0.35, d                    # measured 0.24 on |logp| <= 32.7
    assert min(overlap) >= 22, overlap    # measured 24-25 of 25


def test_lm_persistent_decode_vs_per_op_chain_batch32():
    """the persistent decode kernel (llm_mega.cu) against the per-op fused chain at the benchmark batch (32 ragged Z10 rows): same
    weights, same bf16 operands, different split-K partition / summation order -> logits after two steps agree to fp32 noise
    amplified by bf16 re-rounding; sampled ids agree for the first steps."""
    from cosyvoice_b200 import synth
    c = bctx()
    sd = lm.synth_state_dict(24)
    c.load_state_dict("llm", sd, cfg=[24])
    inputs = synth.batch32_zero_shot(32)
    B = 32
    tl = [int(i["text"].shape[1] + i["prompt_text"].shape[1]) for i in inputs]
    sl = [int(i["llm_prompt_speech_token"].shape[1]) for i in inputs]
    tt = torch.cat([torch.cat([i["prompt_text"], i["text"]], 1).reshape(-1) for i in inputs])
    ss = torch.cat([i["llm_prompt_speech_token"].reshape(-1) for i in inputs])
    U = torch.rand(16, B, 2, generator=torch.Generator().manual_seed(3)).to(c.device)
    big = torch.full((B,), 10000, dtype=torch.int32, device=c.device)

    def run(mega):
        c.set_option("lm_mega", mega)
        try:
            sess = c.lm_session(B, max(tl) + max(sl) + 64)
            ids = torch.zeros(B, 16, dtype=torch.int32, device=c.device)
            cnt = torch.zeros(B, dtype=torch.int32, device=c.device)
            done = torch.zeros(B, dtype=torch.int32, device=c.device)
            st = torch.cuda.Stream()
            torch.cuda.synchronize()
            with torch.cuda.stream(st):
                c.lm_prefill(sess, tt, tl, ss, sl)
                c.lm_decode(sess, 2, U, big, big, ids, cnt, done)
                lg = c.lm_last_logits(sess, B).cpu()
                c.lm_decode(sess, 6, U, big, big, ids, cnt, done)
                out = (lg, ids.cpu().clone())
            torch.cuda.synchronize()
            c.lm_session_destroy(sess)
            return out
        finally:
            c.set_option("lm_mega", 0)      # the library default
    (la, ia), (lb, ib) = run(1), run(0)
    fin = torch.isfinite(la) & torch.isfinite(lb)
    d = (la - lb)[fin].abs().max().item()
    same2 = int((ia[:, :2] == ib[:, :2]).all(1).sum())
    print(f"[batch-32 decode] max |logit(mega) - logit(per-op chain)| after 2 steps {d:.4g}; rows with identical first two ids {same2}/32")
    assert d < 0.3, d
    # sampled (not argmax) ids: a row changes when the 0.1-level logit difference moves a cumulative-probability boundary across its
    # uniform draw - a few rows out of 32 per two steps (28-30 equal in the runs so far)
    assert same2 >= 26, same2


def test_flow_mel_fullsize(golden):
    g = golden("z10_full")
    c = bctx()
    cfg = flow.FlowCfg()
    sd = weights.synth_state_dict(flow.param_shapes(cfg), 1986, flow.SYNTH_GAINS)
    c.load_state_dict("flow", sd, cfg=[cfg.enc_blocks, cfg.enc_up_blocks, cfg.num_mid_blocks, cfg.n_blocks])
    c.set_cfm_noise(flow.cfm_noise(15000)[0].t().contiguous())
    utt, ids, _ = case()
    toks = torch.cat([utt["flow_prompt_speech_token"].reshape(-1), ids.int()])
    mel, lens = c.flow_inference(toks, [toks.numel()], utt["prompt_speech_feat"][0], [150], utt["flow_embedding"])
    ref = torch.from_numpy(g["mel"])[0].t()
    assert mel.shape == ref.shape == (500, 80)
    dd = (mel.cpu() - ref).abs()
    print(f"[full-size flow, bf16] mel max |d| {dd.max().item():.4g}, mean |d| {dd.mean().item():.4g} on |mel| <= {ref.abs().max().item():.3g}; "
          f"yardstick (oracle under torch CPU bf16 autocast vs fp32): max {float(g['mel_autocast_bf16_max']):.4g}, mean {float(g['mel_autocast_bf16_mean']):.4g}")
    # measured on B200: max 0.035, mean 0.0073 - the same as torch's own bf16 autocast shows against fp32 on this model (0.041 / 0.0077)
    assert dd.max().item() < 0.08 and dd.mean().item() < 0.015, (dd.max().item(), dd.mean().item())


def test_hift_wav_fullsize(golden):
    g = golden("z10_full")
    c = bctx()
    sd = weights.synth_state_dict(hift.param_shapes(), 1986, hift.SYNTH_GAINS)
    c.load_state_dict("hift", sd)
    mel = torch.from_numpy(g["mel"])
    # the oracle's source and waveform for the committed mel, recomputed on the CPU from the seeded noise and pinned to the
    # committed samples (make_golden_full.py stores every PIN_STRIDE-th one)
    wav_ref, src = hift.inference(sd, mel, case()[2])
    src, ref = src.reshape(-1), wav_ref.reshape(-1)
    assert np.abs(src[::PIN_STRIDE].numpy() - g["source_pin"]).max() < 1e-4
    assert np.abs(ref[::PIN_STRIDE].numpy() - g["wav_pin"]).max() < 1e-4
    mel_tm = mel[0].t().contiguous()
    f0 = c.hift_f0(mel_tm, [500]).cpu()
    print(f"[full-size vocoder] f0 max |d| {(f0 - torch.from_numpy(g['f0']).reshape(-1)).abs().max().item():.4g} Hz")
    wav = c.hift_decode(mel_tm, [500], src).cpu()
    d = (wav - ref).abs()
    snr = 10 * torch.log10(ref.pow(2).sum() / (wav - ref).pow(2).sum()).item()
    print(f"[full-size vocoder, ctx precision bf16] wav max |d| {d.max().item():.4g}, rms {d.pow(2).mean().sqrt().item():.4g} on |wav| <= {ref.abs().max().item():.3g}; SNR {snr:.1f} dB")
    # IEEE-half operands (10-bit mantissa, the class of the reference's default TF32 convolutions): measured 1.0e-3 / 54 dB SNR on B200;
    # SURVEY.md §8(c)(ii) asks for <= 2e-3 with the source injected
    assert d.max().item() < 2e-3 and snr > 48.0, (d.max().item(), snr)
