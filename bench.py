#!/usr/bin/env python
"""Benchmark of the CosyVoice2-0.5B hot path (LM decode -> CFM flow -> HiFT vocoder) on B200.

Metric (BASELINE.json): audio-sec/s, CosyVoice2-0.5B zero-shot batch-32, NFE=10 - synthetic data (random-init weights of
the reference architecture, random token / prompt tensors of the Z10 shape, SURVEY.md §8d).  One *step* = one pass of
the whole pipeline over one batch of 32 ragged utterances per GPU.

  python bench.py --gpus 1 --steps 3 --warmup 3            # ours (default)
  python bench.py --impl reference --steps 1 --warmup 0    # the reference's algorithm on the host CPU cores
  python bench.py --dump-outputs DIR                       # also write the last timed step's waveforms to DIR/*.npy, so that
                                                           # two builds can be compared output for output (same seeded inputs)
  torchrun --nnodes=1 --nproc-per-node N bench.py --gpus N ...   (N > 1: one rank per GPU; primary = the same 32 requests
                                                                   sharded over the ranks, "weak" key = 32 requests per rank)

Prints ONE JSON line on rank 0 (contract in the task statement): value = device-resident throughput, e2e = the same
metric through the public API with host buffers (H2D of the request tensors, D2H of the waveforms inside the timed
region), roofline = the dominant kernel family against the measured peaks, cpu_baseline = the oracle port on CPU.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BATCH = 32
TOKEN_RATIO = 5.0          # min_token_text_ratio == max_token_text_ratio => exactly 5 * n_text speech tokens (SURVEY.md §8d)
METRIC = "audio-sec/s, CosyVoice2-0.5B zero-shot batch-32, NFE=10"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], tflops=d.get("bf16_tflops_sustained", d["bf16_tflops"]), source="measured (MEASURED_PEAKS.json, sustained)")
    return dict(hbm_gbs=6650.0, tflops=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows)}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


# ================================================================================================ reference arm (CPU)
_REF_WEIGHTS = {}


def host_threads():
    """Threads the CPU arm may use: the affinity mask, clipped by the cgroup CPU quota, at most 32 (batch-1 decode does not scale
    past that and oversubscribing a quota-limited container is slower than running fewer threads)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(float(q) / float(per))))
    except (OSError, ValueError):
        pass
    return max(1, min(n, 32))


def cpu_reference_sample(full=True, threads=None):
    """The reference's algorithm (oracle port, CPU fp32 torch) on ONE Z10 utterance of the batch-32 workload: LM decode of
    5*n_text tokens with KV cache + RAS sampling, flow (NFE 10, CFG), HiFT.  Returns (audio_seconds, wall_seconds, info)."""
    import torch
    from oracle import flow as oflow, hift as ohift, lm as olm, weights as oweights
    from cosyvoice_b200 import synth
    threads = threads or host_threads()
    torch.set_num_threads(threads)
    NL = 24 if full else 2
    fcfg = oflow.FlowCfg() if full else oflow.FlowCfg(2, 1, 2, 2)
    if full not in _REF_WEIGHTS:                       # generated once per process, outside every timed region
        lsd = olm.synth_state_dict(NL)
        lsd["llm_decoder.bias"][6561:6564] = -1e4
        _REF_WEIGHTS[full] = (lsd, oweights.synth_state_dict(oflow.param_shapes(fcfg), 1986, oflow.SYNTH_GAINS),
                              oweights.synth_state_dict(ohift.param_shapes(), 1986, ohift.SYNTH_GAINS))
    lsd, fsd, hsd = _REF_WEIGHTS[full]
    utt = synth.z10_utterance(0, 50)
    g = torch.Generator().manual_seed(0)
    n_tok = int(50 * TOKEN_RATIO)
    U = torch.rand(n_tok + 1, 2, generator=g)
    t0 = time.perf_counter()
    with torch.inference_mode():
        ids = olm.inference(lsd, utt["text"], utt["prompt_text"], utt["llm_prompt_speech_token"], U, NL, min_ratio=TOKEN_RATIO, max_ratio=TOKEN_RATIO)
        t1 = time.perf_counter()
        mel = oflow.inference(fsd, torch.tensor([ids], dtype=torch.int32), utt["flow_prompt_speech_token"], utt["prompt_speech_feat"],
                              utt["flow_embedding"], fcfg)
        t2 = time.perf_counter()
        noise = torch.randn(1, mel.shape[2] * 480, 9, generator=g)
        wav, _ = ohift.inference(hsd, mel, noise)
        t3 = time.perf_counter()
    audio_s = wav.shape[1] / 24000.0
    info = dict(tokens=len(ids), lm_s=t1 - t0, flow_s=t2 - t1, hift_s=t3 - t2)
    return audio_s, t3 - t0, info


def run_reference(args):
    rank, world, local = dist_env()
    if rank != 0:
        return
    cores = host_threads()
    vals = []
    for _ in range(args.warmup):                       # CPU warm-up (page-in, thread pool): the same code on small modules
        cpu_reference_sample(full=False, threads=cores)
    info = {}
    for _ in range(max(args.steps, 1)):
        a, w, info = cpu_reference_sample(full=not args.small, threads=cores)
        vals.append((a, w))
    audio = sum(a for a, _ in vals)
    wall = sum(w for _, w in vals)
    v = audio / wall
    sample = "1 of the 32 Z10 utterances (50 text tokens -> 250 speech tokens, 10 s of audio) per step: " \
             f"LM {info['lm_s']:.1f}s + flow {info['flow_s']:.1f}s + HiFT {info['hift_s']:.1f}s"
    line = {"metric": METRIC, "value": v, "unit": "audio-sec/s", "n_gpus": 0, "steps": max(args.steps, 1), "warmup": args.warmup,
            "ms_per_step": 1000 * wall / max(args.steps, 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": "CosyVoice2-0.5B zero-shot batch-32 NFE=10 (bounded sample: one utterance per step)",
                       "warmup_note": "CPU warm-up steps run the same code on 2-layer modules (thread pool / page-in only)",
                       "reference_impl": "oracle port of cosyvoice/{llm,flow,hifigan} (torch CPU fp32; /root/reference is absent on the GPU box)"},
            "cpu_baseline": {"value": v, "unit": "audio-sec/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "audio-sec/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def stage_roofline(stats, inputs, pk, nfe=10):
    """Per-stage roofline fractions from SURVEY.md §8(d)'s ALGORITHMIC work (not measured traffic) and the CUDA-event stage times
    of the last timed step: LM decode = bf16 weight stream + KV reads per step over the HBM peak; flow = estimator + encoder dense
    FLOPs over the bf16 tensor peak; HiFT = 2 * 306.2e6 FLOP per mel frame over the tensor peak."""
    tokens, frames = stats["tokens"], stats["mel_frames"]
    B = len(tokens)
    L0 = [1 + int(i["prompt_text"].shape[1]) + int(i["text"].shape[1]) + 1 + int(i["llm_prompt_speech_token"].shape[1]) for i in inputs]
    steps = max(tokens) if tokens else 0
    lm_bytes = 0.0
    for i in range(steps):
        live = [b for b in range(B) if tokens[b] > i]
        lm_bytes += 727.6e6 + sum(12288.0 * (L0[b] + i) for b in live) + len(live) * (896 + 6564) * 4
    lm_roof_ms = lm_bytes / (pk["hbm_gbs"] * 1e9) * 1e3
    flow_flop = 0.0
    for b in range(B):
        T = frames[b] + int(inputs[b]["prompt_speech_feat"].shape[1])            # total mel frames incl. the prompt
        flow_flop += 2.0 * (66.09e6 + 57344.0 * T) * T * 2 * nfe                  # estimator, both CFG branches
        flow_flop += 2.0 * 56.6e6 * (T // 2)                                      # encoder dense part
    flow_roof_ms = flow_flop / (pk["tflops"] * 1e12) * 1e3
    hift_flop = sum(2.0 * 306.2e6 * f for f in frames)
    hift_roof_ms = hift_flop / (pk["tflops"] * 1e12) * 1e3
    out = {}
    for name, roof, meas, bound in (("lm", lm_roof_ms, stats["lm_ms"], "hbm"), ("flow", flow_roof_ms, stats["flow_ms"], "tensor"),
                                    ("hift", hift_roof_ms, stats["hift_ms"], "tensor")):
        out[name] = {"bound": bound, "roofline_ms": round(roof, 3), "measured_ms": round(meas, 3), "frac": round(roof / meas, 4) if meas > 0 else None}
    out["lm"]["decode_steps"] = steps
    return out


DUMP_BYTES = 64_000_000


def dump_outputs(path, outputs, rank, world):
    """--dump-outputs: what the last timed tts_batch_device call returned, as .npy files - wav (float32, the utterances' samples
    back to back) and lens (float64, samples per utterance), with a _rank<r> suffix when several ranks run.  A waveform larger
    than its rank's share of 64 MB is written as every k-th sample, k the smallest stride that fits."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    suffix = f"_rank{rank}" if world > 1 else ""
    wav, lens = outputs["wav"].numpy(), outputs["lens"].numpy()
    cap = (DUMP_BYTES // world - lens.nbytes) // wav.itemsize
    np.save(os.path.join(path, f"wav{suffix}.npy"), wav[::max(1, -(-wav.size // cap))])
    np.save(os.path.join(path, f"lens{suffix}.npy"), lens)


# ================================================================================================ our arm (GPU)
def run_ours(args):
    import torch
    rank, world, local = dist_env()
    n_gpus = args.gpus
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        dist = None
    from cosyvoice_b200 import synth
    from cosyvoice_b200.model import B200CosyVoice2Model
    from cosyvoice_b200.parallel import broadcast_state_dicts, gather_flat, shard_lpt
    dev = torch.device("cuda", local)
    full = not args.small
    nl, fcfg = (24, (6, 4, 12, 4)) if full else (2, (2, 1, 2, 2))
    # weights: rank 0 draws them, NCCL broadcast to the other ranks (the only weight traffic of the job)
    sds = synth.cosyvoice2_state_dicts(dev, 1986, nl, fcfg) if rank == 0 else None
    sds = broadcast_state_dicts(sds, dev, synth.llm_shapes(nl), synth.flow_shapes(*fcfg), synth.hift_shapes(), dist)
    model = B200CosyVoice2Model(precision=args.precision, device=local, workspace_gb=args.workspace_gb)
    model.load_state_dicts(*sds)
    del sds
    torch.cuda.empty_cache()
    model.min_token_text_ratio = model.max_token_text_ratio = TOKEN_RATIO
    model.lm_chains = args.lm_chains
    for kv in args.opt:                                # debug/experiment switches of the library (cvk_set_option)
        k, v = kv.split("=")
        model.ctx.set_option(k, int(v))
    batch = args.batch

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def measure(inputs, counts, want_clocks):
        """K timed steps device-resident (`value`) + K timed steps end to end (`e2e`: pinned host inputs -> H2D inside the step ->
        pipeline -> device-resident gather of every rank's waveform buffer on rank 0 -> one pinned D2H)."""
        inputs_dev = [{k: v.to(dev) for k, v in i.items()} for i in inputs]
        pinned = [{k: v.pin_memory() for k, v in i.items()} for i in inputs]
        h2d = sum(sum(v.numel() * v.element_size() for v in i.values()) for i in inputs)
        for _ in range(args.warmup):
            model.tts_batch_device(inputs_dev)
        # ---- timed region 1: inputs resident in HBM, waveforms left in HBM, no per-launch instrumentation
        sampler = ClockSampler(local)
        barrier()
        if rank == 0 and want_clocks:
            sampler.start()
        l0 = model.ctx.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(model.stream)
        audio_s, stats = 0.0, None
        for _ in range(args.steps):
            wav, n, stats = model.tts_batch_device(inputs_dev)
            audio_s += sum(n) / 24000.0
        e1.record(model.stream)
        barrier()
        dev_ms = e0.elapsed_time(e1)
        wall_ms = 1000 * (time.perf_counter() - t0)
        launches = model.ctx.launch_count() - l0
        clocks = sampler.stop() if (rank == 0 and want_clocks) else None
        stats = model._stage_ms(stats)
        outputs = dict(wav=wav.cpu(), lens=torch.tensor(n, dtype=torch.float64)) if args.dump_outputs else None
        # ---- timed region 2: end to end through the public API
        with torch.cuda.stream(model.stream):
            wav, n, _ = model.tts_batch_device(pinned)
            gather_flat(wav, [k for k in n if k], dist, dev, counts)        # untimed: NCCL sets up its point-to-point channels on first use
        barrier()
        t0 = time.perf_counter()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record(model.stream)
        audio_e2e, d2h = 0.0, 0
        for _ in range(args.steps):
            with torch.cuda.stream(model.stream):
                wav, n, _ = model.tts_batch_device(pinned)
                got = gather_flat(wav, [k for k in n if k], dist, dev, counts)
            audio_e2e += sum(n) / 24000.0
            if got is not None:
                d2h = got[0].numel() * 4
        f1.record(model.stream)
        barrier()
        e2e_ms = max(f0.elapsed_time(f1), 1000 * (time.perf_counter() - t0))
        # ---- max over ranks, totals over ranks
        tt = torch.tensor([dev_ms, e2e_ms, wall_ms], device=dev, dtype=torch.float64)
        aa = torch.tensor([audio_s, audio_e2e, float(launches), float(h2d)], device=dev, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dist.all_reduce(aa, op=dist.ReduceOp.SUM)
        dev_ms, e2e_ms, wall_ms = tt.tolist()
        audio_s, audio_e2e, launches, h2d_all = aa.tolist()
        return dict(value=audio_s / (dev_ms / 1000.0), e2e=audio_e2e / (e2e_ms / 1000.0), dev_ms=dev_ms, e2e_ms=e2e_ms, wall_ms=wall_ms,
                    launches=int(launches), h2d=int(h2d_all), d2h=int(d2h), clocks=clocks, stats=stats, inputs=inputs, outputs=outputs)

    # ---- primary: the contract's split - the SAME `batch` utterances sharded over the ranks (strong scaling), LPT on expected tokens
    all_inputs = synth.batch32_zero_shot(batch)
    plan = shard_lpt([int(i["text"].shape[1] * TOKEN_RATIO) for i in all_inputs], world)
    strong = measure([all_inputs[i] for i in plan[rank]], [len(p) for p in plan], True)
    # ---- one extra instrumented step (CUDA events around every GEMM / attention launch) for the per-family roofline
    model.ctx.profile(1)
    model.tts_batch_device([{k: v.to(dev) for k, v in i.items()} for i in strong["inputs"]])
    torch.cuda.synchronize()
    prof = [model.ctx.profile_read(f) for f in range(3)]
    model.ctx.profile(0)
    # ---- secondary: weak scaling (every rank its own `batch` requests)
    weak = measure(synth.batch32_zero_shot(batch, base=rank * batch), [batch] * world, False) if world > 1 else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, strong["outputs"], rank, world)
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    pk = peaks()
    value, e2e_v, dev_ms = strong["value"], strong["e2e"], strong["dev_ms"]
    # dominant kernel family = the one with the largest share of device time (instrumented step)
    fam_names = ["conv_gemm_tc (tcgen05 bf16)", "conv_gemm_simt (fp32 CUDA cores)", "attention (tcgen05 flash kernels; fp32-math CUDA-core kernel in fp32 mode)"]
    dom = max(range(3), key=lambda f: prof[f]["ms"])
    p = prof[dom]
    ach = p["flops"] / (p["ms"] / 1000.0) / 1e12 if p["ms"] > 0 else 0.0
    roof = {"bound": "tensor", "achieved": ach, "peak": pk["tflops"], "unit": "TFLOP/s", "frac": ach / pk["tflops"]}
    traffic, traffic_note = None, "no ncu capture committed for this kernel"
    for name in ("r02_traffic.json", "r01_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", name)
        if dom == 0 and os.path.exists(tpath):            # dram__bytes_read.sum + dram__bytes_write.sum of ONE launch from `ncu --set full`
            tj = json.load(open(tpath))
            traffic, traffic_note = tj["dram_bytes_per_launch"], tj["note"]
            break
    step_ms = dev_ms / args.steps
    roof.update({"traffic": traffic, "traffic_note": traffic_note, "kernel": fam_names[dom], "launches": p["launches"], "avg_launch_ms": p["ms"] / max(p["launches"], 1),
                 "share_of_step": p["ms"] / step_ms, "peak_source": pk["source"], "timed": "one extra instrumented step (not inside the `value` region)",
                 "families_ms": {fam_names[f]: prof[f]["ms"] for f in range(3)}})
    cpu = None
    if n_gpus == 1 and not args.no_cpu_baseline:
        a, w, info = cpu_reference_sample(full=full)
        cpu = {"value": a / w, "unit": "audio-sec/s", "cores": host_threads(), "kind": "port",
               "sample": f"1 of the {batch} utterances (250 speech tokens, 10 s audio): LM {info['lm_s']:.1f}s flow {info['flow_s']:.1f}s HiFT {info['hift_s']:.1f}s"}
    stats = strong["stats"]
    per_gpu = [len(pl) for pl in plan]
    line = {"metric": METRIC, "value": value, "unit": "audio-sec/s", "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": step_ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
            "config": {"workload": f"CosyVoice2-0.5B zero-shot batch-{batch} (the same {batch} ragged Z10 requests sharded over the GPUs by LPT on expected tokens: "
                                   f"{per_gpu} per GPU), NFE=10, 40-60 text tokens -> 200-300 speech tokens, 75 prompt tokens / 150 prompt mel frames"
                                   + ("" if full else " [SMALL DEBUG MODEL]"),
                       "global_batch": batch, "per_gpu": per_gpu, "nfe": 10,
                       "l2": "working set (1.3 GB weights + GBs of activations) exceeds the 126 MB L2",
                       "parallelism": f"dp{n_gpus} (independent utterances, weights broadcast once over NCCL, waveform buffers gathered device-to-device on rank 0)",
                       "stage_ms_last_step_rank0": {k: stats[k] for k in ("lm_ms", "flow_ms", "hift_ms")}, "rtf": 1.0 / value},
            "e2e": {"value": e2e_v, "unit": "audio-sec/s", "h2d_bytes_per_step": strong["h2d"], "d2h_bytes_per_step": strong["d2h"]},
            "gpu_launches": strong["launches"], "clocks": strong["clocks"], "roofline": roof, "wall_ms_per_step": strong["wall_ms"] / args.steps}
    try:                                                # per-stage view the north star asks for; never allowed to break the line
        line["stage_roofline"] = stage_roofline(stats, strong["inputs"], pk)
        lim = max(("lm", "flow", "hift"), key=lambda k: stats[k + "_ms"])
        line["stage_roofline"]["limiting_stage_rank0"] = lim
    except Exception as e:                              # noqa: BLE001
        line["stage_roofline"] = {"error": repr(e)}
    if weak is not None:
        line["weak"] = {"value": weak["value"], "unit": "audio-sec/s", "ms_per_step": weak["dev_ms"] / args.steps, "e2e": weak["e2e"],
                        "workload": f"{batch} requests PER GPU ({batch * world} in flight)",
                        "stage_ms_last_step_rank0": {k: weak["stats"][k] for k in ("lm_ms", "flow_ms", "hift_ms")}}
    if cpu:
        line["cpu_baseline"] = cpu
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


# ================================================================================================ config #4: CosyVoice3 bi-streaming
def run_cv3_bistream(args):
    """BASELINE.json configs[3]: Fun-CosyVoice3-0.5B bi-streaming (text arrives as a generator, audio leaves in chunks), batch 8 on
    one GPU: 8 concurrent tts(text=<generator>, stream=True) requests on ONE B200CosyVoice3Model (the reference serves concurrent
    requests from threads, runtime/python/grpc/server.py:69).  Every yielded chunk is a host tensor, so `value` and `e2e` are the
    same measurement here (the public API has no device-resident variant of a streaming request)."""
    import threading
    import torch
    from cosyvoice_b200 import synth
    from cosyvoice_b200.model3 import B200CosyVoice3Model
    dev = torch.device("cuda", 0)
    full = not args.small
    nl, depth = (24, 22) if full else (2, 2)
    model = B200CosyVoice3Model(precision=args.precision, device=0, workspace_gb=args.workspace_gb)
    model.load_state_dicts(*synth.cosyvoice3_state_dicts(dev, 1986, nl, depth))
    torch.cuda.empty_cache()
    model.silent_tokens = []                   # uniform synthetic ids: count every id
    batch = args.batch if args.batch != BATCH else 8
    reqs = [synth.cv3_bistream_request(i) for i in range(batch)]
    model.bistream_max_tokens = int(reqs[0]["text"].shape[1] * TOKEN_RATIO)          # random weights never emit eos (see model.py)
    pinned = [{k: (v.pin_memory() if torch.is_tensor(v) else [c.pin_memory() for c in v]) for k, v in r.items()} for r in reqs]
    h2d = sum(sum(v.numel() * v.element_size() for v in r.values() if torch.is_tensor(v)) for r in reqs)

    def one(r, out, i):
        n, first = 0, None
        t0 = time.perf_counter()
        for o in model.tts(text=iter(r["text_chunks"]), flow_embedding=r["flow_embedding"], llm_embedding=r["llm_embedding"],
                           prompt_text=r["prompt_text"], llm_prompt_speech_token=r["llm_prompt_speech_token"],
                           flow_prompt_speech_token=r["flow_prompt_speech_token"], prompt_speech_feat=r["prompt_speech_feat"], stream=True):
            if first is None:
                first = time.perf_counter() - t0
            n += o["tts_speech"].shape[1]
        out[i] = (n, first)

    def step():
        model.token_hop_len = 25
        out = [None] * batch
        ts = [threading.Thread(target=one, args=(pinned[i], out, i)) for i in range(batch)]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        return out
    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(0)
    torch.cuda.synchronize()
    sampler.start()
    l0 = model.ctx.launch_count()
    t0 = time.perf_counter()
    audio, firsts, d2h = 0.0, [], 0
    for _ in range(args.steps):
        out = step()
        audio += sum(n for n, _ in out) / 24000.0
        firsts += [f for _, f in out]
        d2h = sum(n for n, _ in out) * 4
    torch.cuda.synchronize()
    wall_ms = 1000 * (time.perf_counter() - t0)
    clocks = sampler.stop()
    launches = model.ctx.launch_count() - l0
    v = audio / (wall_ms / 1000.0)
    firsts.sort()
    line = {"metric": "audio-sec/s, Fun-CosyVoice3-0.5B bi-streaming batch-8, NFE=10", "value": v, "unit": "audio-sec/s", "n_gpus": 1, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": wall_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
            "config": {"workload": f"Fun-CosyVoice3-0.5B bi-streaming: {batch} concurrent tts(text generator of 4 chunks, stream=True) requests, 48 text ids -> "
                                   f"{model.bistream_max_tokens} speech ids each (capped: random weights emit no eos), 75 prompt tokens / 150 prompt mel frames, DiT depth {depth}, "
                                   "causal vocoder; chunk schedule hop 25 -> 50 -> 100 with 3 look-ahead tokens (cli/model.py:346-373)" + ("" if full else " [SMALL DEBUG MODEL]"),
                       "batch": batch, "nfe": 10, "first_chunk_latency_s": {"median": firsts[len(firsts) // 2], "max": firsts[-1]},
                       "timing": "wall clock around the concurrent requests (every chunk is a host tensor; no device-only variant of the streaming API)"},
            "e2e": {"value": v, "unit": "audio-sec/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches), "clocks": clocks}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--small", action="store_true", help="debug: 2-layer LM / reduced flow (NOT the benchmark config)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workspace-gb", type=float, default=40.0)
    ap.add_argument("--lm-chains", type=int, default=1)
    ap.add_argument("--opt", action="append", default=[], help="library option key=value (cvk_set_option), repeatable")
    ap.add_argument("--workload", default="batch32", choices=["batch32", "cv3-bistream"],
                    help="batch32 = the headline metric (BASELINE.json configs[2]); cv3-bistream = configs[3] (1 GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="batch32 on the GPU: write the waveforms of the last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "batch32"):
        ap.error("--dump-outputs applies to the batch32 workload of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "cv3-bistream":
        run_cv3_bistream(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
