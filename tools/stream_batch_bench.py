"""Batched streaming synthesis against one thread per stream.  Full-size random-init CosyVoice2 (bf16), N Z10-shaped streaming
requests (75 prompt tokens, 50 text ids -> exactly 250 speech ids, min = max token ratio 5 as in bench.py), N in --n.  Two arms in
the same process, alternating:
  (a) N threads, each calling tts(stream=True) on the shared model (the reference's serving pattern; every chunk is its own flow
      call under the context lock);
  (b) one tts_stream_batch of the N requests (one multi-slot flow session, one chunk_batch call per round).
Reports first-chunk latency (median / max over requests), the gaps between a request's chunks, audio-s/s over all streams, flow
calls and cvk_launch_count per step, and the card name and power limit read in the same run.  An untimed check compares the arms'
outputs on the same seeds (per-request uniforms; vocoder noise seeded by chunk length).  Prints one JSON line."""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from cosyvoice_b200 import synth  # noqa: E402
from cosyvoice_b200.model import B200CosyVoice2Model  # noqa: E402

RATIO = 5.0


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                            timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unavailable"
    return {"name": name, "power_limit": pl}


def stats(xs):
    xs = sorted(xs)
    return {"median": xs[len(xs) // 2], "max": xs[-1]} if xs else None


class Counter:
    """counts the flow calls a step makes (chunk calls on sessions, prefix / final flow calls)"""

    def __init__(self, ctx):
        self.n = {}
        for name in ("flow_stream_chunk", "flow_stream_chunk_batch", "flow_inference"):
            fn = getattr(ctx, name)
            setattr(ctx, name, self._wrap(name, fn))

    def _wrap(self, name, fn):
        def w(*a, **k):
            self.n[name] = self.n.get(name, 0) + 1
            return fn(*a, **k)
        return w


def arm_threads(m, reqs):
    t0 = time.perf_counter()
    times = [[] for _ in reqs]
    audio = [0] * len(reqs)

    def one(i):
        for o in m.tts(**reqs[i], stream=True):
            times[i].append(time.perf_counter() - t0)
            audio[i] += o["tts_speech"].shape[1]
    m.token_hop_len = 25
    ts = [threading.Thread(target=one, args=(i,)) for i in range(len(reqs))]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    return time.perf_counter() - t0, times, audio


def arm_batch(m, reqs):
    t0 = time.perf_counter()
    times = [[] for _ in reqs]
    audio = [0] * len(reqs)
    for i, o, _ in m.tts_stream_batch(reqs):
        times[i].append(time.perf_counter() - t0)
        audio[i] += o["tts_speech"].shape[1]
    return time.perf_counter() - t0, times, audio


def agreement(m, reqs):
    """same seeds through both paths: per-request uniforms, vocoder noise a function of the chunk's sample count"""
    d = m.device
    steps = int(reqs[0]["text"].shape[1] * RATIO) + 1
    g = torch.Generator().manual_seed(11)
    U = torch.rand(steps, len(reqs), 2, generator=g)

    def noise(n):
        gg = torch.Generator(device=d)
        gg.manual_seed(n)
        return torch.randn(n, 9, device=d, generator=gg)
    m.noise_fn = noise
    try:
        batch = [[] for _ in reqs]
        for i, o, _ in m.tts_stream_batch(reqs, uniforms=U):
            batch[i].append(o["tts_speech"])
        out = {"chunk_lens_equal": True, "max_abs_diff": 0.0}
        for i, r in enumerate(reqs):
            m.token_hop_len = 25
            m.uniforms_override = U[:, i:i + 1].contiguous()
            alone = [o["tts_speech"] for o in m.tts(**r, stream=True)]
            if [c.shape[1] for c in alone] != [c.shape[1] for c in batch[i]]:
                out["chunk_lens_equal"] = False
                continue
            out["max_abs_diff"] = max(out["max_abs_diff"], (torch.cat(alone, 1) - torch.cat(batch[i], 1)).abs().max().item())
        return out
    finally:
        m.noise_fn, m.uniforms_override = None, None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", default="1,4,8,16", help="comma-separated stream counts")
    ap.add_argument("--steps", type=int, default=2, help="timed steps per arm and N (after one warm-up step each)")
    ap.add_argument("--small", action="store_true", help="debug: 2-layer LM / reduced flow (NOT the measurement config)")
    ap.add_argument("--workspace-gb", type=float, default=40.0)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("stream_batch_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    nl, fcfg = (2, (2, 1, 2, 2)) if a.small else (24, (6, 4, 12, 4))
    m = B200CosyVoice2Model(precision="bf16", device=0, workspace_gb=a.workspace_gb)
    m.load_state_dicts(*synth.cosyvoice2_state_dicts(dev, 1986, nl, fcfg))
    torch.cuda.empty_cache()
    m.min_token_text_ratio = m.max_token_text_ratio = RATIO
    # both arms cache the same frames per stream: prompt + every generated token (the default 2048 would hold 16 one-slot sessions
    # of 4.7 GB each in arm (a))
    m.stream_cache_frames = 2 * (75 + 250)
    cnt = Counter(m.ctx)
    ns = [int(x) for x in a.n.split(",")]
    res = {"card": card(), "arms": {}}
    for N in ns:
        reqs = [synth.z10_utterance(i, 50) for i in range(N)]
        rows = {}
        for name, fn in (("a_threads", arm_threads), ("b_stream_batch", arm_batch)):
            fn(m, reqs)                                            # warm-up
            rows[name] = {"first_chunk_s": [], "gap_s": [], "audio_s": 0.0, "wall_s": 0.0, "flow_calls": {}, "launches": 0}
        for _ in range(a.steps):
            for name, fn in (("a_threads", arm_threads), ("b_stream_batch", arm_batch)):
                r = rows[name]
                cnt.n = {}
                torch.cuda.synchronize()
                l0 = m.ctx.launch_count()
                wall, times, audio = fn(m, reqs)
                torch.cuda.synchronize()
                r["launches"] += (m.ctx.launch_count() - l0) / a.steps
                for k, v in cnt.n.items():
                    r["flow_calls"][k] = r["flow_calls"].get(k, 0) + v / a.steps
                r["first_chunk_s"] += [t[0] for t in times]
                r["gap_s"] += [y - x for t in times for x, y in zip(t, t[1:])]
                r["audio_s"] += sum(audio) / 24000.0
                r["wall_s"] += wall
        for name, r in rows.items():
            rows[name] = {"first_chunk_s": stats(r["first_chunk_s"]), "chunk_gap_s": stats(r["gap_s"]),
                          "audio_s_per_s": r["audio_s"] / r["wall_s"], "flow_calls_per_step": r["flow_calls"],
                          "launches_per_step": r["launches"]}
        rows["agreement"] = agreement(m, reqs)
        res["arms"][str(N)] = rows
        print(f"N={N}: " + json.dumps(rows), file=sys.stderr)
    res["config"] = ("CosyVoice2-0.5B random-init bf16" + (" [SMALL DEBUG MODEL]" if a.small else "") +
                     f"; Z10 requests (75 prompt tokens, 50 text ids -> 250 speech ids); {a.steps} timed steps per arm after 1 warm-up; "
                     "wall clock from the start of a step to each yielded chunk (chunks are host tensors)")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
