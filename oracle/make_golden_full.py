"""Golden outputs AT THE BENCHMARK SHAPE (one full-size Z10 utterance: 24-layer LM, 650-frame flow, 500-frame vocoder) for the
bf16-mode parity tests (tests/test_zz_fullsize_gpu.py).  TEST INFRASTRUCTURE: CPU oracle only (the oracle itself is pinned against
the unmodified reference at small sizes by oracle/make_golden.py; the full-size run here is the same functions on the same
synthetic-weight recipe, ~3 CPU-minutes).

  python -m oracle.make_golden_full        -> tests/golden/z10_full.npz

Contents: LM teacher-forced log-probs of 8 positions (over 139 prompt + 250 speech-token positions, 24 layers), the flow's mel
[80, 500] for those 250 tokens (prompt 75 tokens / 150 frames, NFE 10, CFG 0.7), the vocoder's f0 for that mel, and every
PIN_STRIDE-th sample of its source and waveform.  The vocoder takes seconds on the CPU, so the test recomputes the full source and
waveform from the committed mel and the seeded noise of case(), and checks them against these samples; storing them in full would
take 1.8 MB."""
import os
import sys
import time

import numpy as np
import torch
import torch.nn.functional as F

from . import flow, hift, lm, weights
from cosyvoice_b200 import synth

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "z10_full.npz")
LM_ROWS = (0, 35, 70, 105, 140, 175, 210, 249)          # offsets into the 250 teacher-forced positions
PIN_STRIDE = 16                                          # stored samples of the vocoder's source and waveform


def case():
    utt = synth.z10_utterance(0, 50)
    g = torch.Generator().manual_seed(2024)
    ids = torch.randint(0, 6561, (250,), generator=g)
    noise = torch.randn(1, 500 * 480, 9, generator=g)
    return utt, ids, noise


@torch.inference_mode()
def main():
    torch.set_num_threads(min(32, os.cpu_count() or 1))
    utt, ids, noise = case()
    t0 = time.time()
    lsd = lm.synth_state_dict(24)
    lm_in = lm.build_lm_input(lsd, utt["text"], utt["prompt_text"], utt["llm_prompt_speech_token"])
    full = torch.cat([lm_in, F.embedding(ids[None], lsd["speech_embedding.weight"])], 1)
    y, _ = lm.qwen2_forward(lsd, full, None, 24)
    L0 = lm_in.shape[1]
    rows = [L0 - 1 + r for r in LM_ROWS]               # position L0-1+r predicts teacher-forced token r
    logp = lm.logprobs(lsd, y[0, rows]).float()
    print(f"lm: {full.shape[1]} positions, {time.time() - t0:.1f}s, |logp| max {logp.abs().max():.3g}")
    del lsd, y
    t0 = time.time()
    fcfg = flow.FlowCfg()
    fsd = weights.synth_state_dict(flow.param_shapes(fcfg), 1986, flow.SYNTH_GAINS)
    mel = flow.inference(fsd, ids[None].int(), utt["flow_prompt_speech_token"], utt["prompt_speech_feat"], utt["flow_embedding"], fcfg)
    print(f"flow: mel {tuple(mel.shape)}, {time.time() - t0:.1f}s, |mel| max {mel.abs().max():.3g}")
    # yardstick (SURVEY.md §8c iii): the same computation under torch's own 16-bit autocast (what the reference's fp16=True mode
    # does to the flow, cli/model.py:293) against fp32 - the deviation a reduced-precision-operand implementation is expected to show
    with torch.autocast("cpu", dtype=torch.bfloat16):
        mel_ac = flow.inference(fsd, ids[None].int(), utt["flow_prompt_speech_token"], utt["prompt_speech_feat"], utt["flow_embedding"], fcfg)
    ac = (mel_ac.float() - mel).abs()
    print(f"flow under CPU bf16 autocast vs fp32: max |d| {ac.max():.3g}, mean |d| {ac.mean():.3g}")
    del fsd
    t0 = time.time()
    hsd = weights.synth_state_dict(hift.param_shapes(), 1986, hift.SYNTH_GAINS)
    f0 = hift.f0_predict(hsd, mel)
    wav, src = hift.inference(hsd, mel, noise)
    print(f"hift: wav {tuple(wav.shape)}, {time.time() - t0:.1f}s, |wav| max {wav.abs().max():.3g}")
    np.savez_compressed(OUT, mel_autocast_bf16_max=np.float32(ac.max()), mel_autocast_bf16_mean=np.float32(ac.mean()), lm_logp=logp.numpy(), lm_rows=np.array(LM_ROWS), ids=ids.numpy().astype(np.int32), mel=mel.numpy(),
                        f0=f0.numpy(), source_pin=src.numpy().reshape(-1)[::PIN_STRIDE].astype(np.float32),
                        wav_pin=wav.numpy().reshape(-1)[::PIN_STRIDE])
    print("wrote", OUT, os.path.getsize(OUT) // 1024, "KiB")


if __name__ == "__main__":
    main()
