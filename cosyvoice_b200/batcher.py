"""Continuous batching in front of ``tts_batch`` + the reference servers' wire format (SURVEY.md §8(f) rank 3).

The reference serves one request per thread: every FastAPI / gRPC handler calls ``cosyvoice.inference_*`` itself and streams
``(tts_speech.numpy() * 2**15).astype(np.int16).tobytes()`` back (runtime/python/fastapi/server.py:40-43,
runtime/python/grpc/server.py:62-64).  On a B200 a single utterance leaves the GPU launch-bound, while the batched pipeline
(``B200CosyVoice2Model.tts_batch``) is what the headline metric measures - so the step after the hot path is a queue that turns
concurrent requests into ragged batches.  This module is that queue and nothing else: no HTTP / gRPC layer, no text
normalisation, no tokenizer (those stay with the reference's frontend and server code, which call ``submit`` instead of
``model.tts``).

Admission policy: a batch is closed when ``max_batch`` requests are waiting or ``max_wait_ms`` have passed since the first one
arrived; requests are never reordered inside a batch (the model's RNG streams are consumed in input order, so a fixed arrival
order gives fixed results).  One worker thread owns the model; ``tts_batch`` itself is ragged, so no padding or bucketing is
needed here.  Streaming requests (``submit_stream``) share the queue: a closed batch serves its streaming requests through one
``tts_stream_batch`` and its offline requests through one ``tts_batch``.  A request never joins a batch that is already running.
"""
import queue
import threading
import time
from concurrent.futures import Future

import numpy as np


def pcm16(wave):
    """float waveform tensor / array in [-1, 1) -> little-endian int16 PCM bytes, the reference servers' wire format
    (runtime/python/fastapi/server.py:42: ``(i['tts_speech'].numpy() * (2 ** 15)).astype(np.int16).tobytes()``, same expression in
    grpc/server.py:64).  Like the reference there is no clipping: callers own the [-1, 1) range (the vocoder clamps to 0.99,
    hifigan/generator.py:566)."""
    a = wave.detach().cpu().numpy() if hasattr(wave, "detach") else np.asarray(wave)
    return (a * (2 ** 15)).astype(np.int16).tobytes()


def pcm16_decode(buf):
    """int16 PCM bytes -> float32 [1, N] in [-1, 1): how the gRPC server reads a prompt waveform from the request
    (runtime/python/grpc/server.py:45-46: ``np.frombuffer(..., dtype=np.int16)`` then ``.float() / (2 ** 15)``)."""
    import torch
    return torch.from_numpy(np.array(np.frombuffer(buf, dtype=np.int16))).unsqueeze(0).float() / (2 ** 15)


class ChunkStream:
    """Iterator over one streaming request's chunks, fed by the batcher's worker: [1, n] float32 CPU tensors, or int16 PCM bytes
    for ``submit_stream_pcm``.  Ends after the request's last chunk; raises the batch's exception if its batch failed."""

    def __init__(self, pcm):
        self.pcm = pcm
        self._q = queue.Queue()
        self._end = None

    def _put(self, wave):
        self._q.put((0, pcm16(wave) if self.pcm else wave))

    def _finish(self, exc=None):
        self._q.put((1, exc))

    def __iter__(self):
        return self

    def __next__(self):
        if self._end is None:
            kind, v = self._q.get()
            if kind == 0:
                return v
            self._end = (v,)
        if self._end[0] is not None:
            raise self._end[0]
        raise StopIteration


class TtsBatcher:
    """``submit(**tts_kwargs)`` -> Future of the waveform ([1, N] float32 CPU tensor, what ``tts`` yields for stream=False);
    ``submit_pcm`` -> Future of the int16 PCM bytes.  ``tts_kwargs`` are the keyword arguments of ``CosyVoice2Model.tts`` that the
    batched pipeline consumes: text, prompt_text, llm_prompt_speech_token, flow_prompt_speech_token, prompt_speech_feat,
    flow_embedding."""

    def __init__(self, model, max_batch=32, max_wait_ms=10.0):
        assert max_batch >= 1
        self.model = model
        self.max_batch = int(max_batch)
        self.max_wait = float(max_wait_ms) / 1e3
        self._q = []                       # (request dict, Future, wants_pcm)
        self._cv = threading.Condition()
        self._closed = False
        self.batches = []                  # sizes of the batches run so far (observability / tests)
        self._worker = threading.Thread(target=self._run, name="cvk-batcher", daemon=True)
        self._worker.start()

    # ------------------------------------------------------------------ client side
    def submit(self, **request):
        return self._enqueue(request, False)

    def submit_pcm(self, **request):
        return self._enqueue(request, True)

    def submit_stream(self, **request):
        """-> iterator of the request's chunks ([1, n] float32 CPU tensors, what ``tts(stream=True)`` yields for it alone)"""
        return self._enqueue(request, False, ChunkStream(False))

    def submit_stream_pcm(self, **request):
        """-> iterator of the request's chunks as int16 PCM bytes (the reference servers' per-chunk wire format)"""
        return self._enqueue(request, True, ChunkStream(True))

    def _enqueue(self, request, pcm, sink=None):
        sink = sink if sink is not None else Future()
        with self._cv:
            if self._closed:
                raise RuntimeError("TtsBatcher is closed")
            self._q.append((request, sink, pcm, time.monotonic()))
            self._cv.notify_all()
        return sink

    def close(self, wait=True):
        """Stop admitting; requests already queued are still served."""
        with self._cv:
            self._closed = True
            self._cv.notify_all()
        if wait:
            self._worker.join()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ------------------------------------------------------------------ worker
    def _take_batch(self):
        with self._cv:
            while not self._q and not self._closed:
                self._cv.wait()
            if not self._q:
                return None
            deadline = self._q[0][3] + self.max_wait
            while len(self._q) < self.max_batch and not self._closed:
                left = deadline - time.monotonic()
                if left <= 0:
                    break
                self._cv.wait(left)
            batch, self._q = self._q[:self.max_batch], self._q[self.max_batch:]
            return batch

    def _run(self):
        while True:
            batch = self._take_batch()
            if batch is None:
                return
            live = [b for b in batch if isinstance(b[1], ChunkStream) or b[1].set_running_or_notify_cancel()]
            if not live:
                continue
            self.batches.append(len(live))
            streams = [b for b in live if isinstance(b[1], ChunkStream)]
            offline = [b for b in live if not isinstance(b[1], ChunkStream)]
            # the kind that arrived first is served first
            for group in sorted((g for g in (streams, offline) if g), key=lambda g: g[0][3]):
                if group is streams:
                    self._serve_streams(streams)
                else:
                    self._serve_offline(offline)

    def _serve_offline(self, live):
        try:
            waves = self.model.tts_batch([b[0] for b in live])
        except BaseException as e:          # the whole batch shares the failure (one launch sequence)
            for _, fut, _, _ in live:
                fut.set_exception(e)
            return
        for (_, fut, pcm, _), w in zip(live, waves):
            try:
                fut.set_result(pcm16(w) if pcm else w)
            except BaseException as e:
                fut.set_exception(e)

    def _serve_streams(self, live):
        open_ = set(range(len(live)))
        try:
            for i, out, last in self.model.tts_stream_batch([b[0] for b in live]):
                live[i][1]._put(out["tts_speech"])
                if last:
                    live[i][1]._finish()
                    open_.discard(i)
        except BaseException as e:          # the failure reaches every request of this batch that has not ended
            for i in sorted(open_):
                live[i][1]._finish(e)
            return
        for i in sorted(open_):
            live[i][1]._finish(RuntimeError("tts_stream_batch ended without the request's last chunk"))
