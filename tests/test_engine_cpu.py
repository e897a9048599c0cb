"""Host-side protocol of the drop-in boundary (no GPU): the LM worker queue
(launch_thread_safe_queue, inference.py:736-799) and TTSInferenceEngine.inference
(inference_engine/__init__.py:40-142) with the device work replaced by stand-ins."""
import json
import queue
from pathlib import Path

import numpy as np
import pytest
import torch

import fish_speech_b200.models.text2semantic.inference as inf
from fish_speech_b200.inference_engine import TTSInferenceEngine
from fish_speech_b200.inference_engine.schema import ServeTTSRequest
from fish_speech_b200.models.dac.modded_dac import DAC


class _FakeModel:
    class config:
        max_seq_len = 64

    dtype = torch.bfloat16

    def setup_caches(self, **kw):
        self.caches = kw


def _fake_generate_long(*, model, decode_one_token, text, **kw):
    if text == "boom":
        raise ValueError("bad request")
    yield inf.GenerateResponse(action="sample", codes=torch.zeros(10, 3, dtype=torch.long), text=text)
    yield inf.GenerateResponse(action="next")


def test_worker_queue_protocol(monkeypatch):
    monkeypatch.setattr(inf, "init_model", lambda *a, **k: (_FakeModel(), inf.decode_one_token_ar))
    monkeypatch.setattr(inf, "generate_long", _fake_generate_long)
    q = inf.launch_thread_safe_queue("ckpt", "cpu", torch.bfloat16)
    rq = queue.Queue()
    q.put(inf.GenerateRequest(request=dict(text="hello"), response_queue=rq))
    a, b = rq.get(timeout=10), rq.get(timeout=10)
    assert a.status == "success" and a.response.action == "sample" and a.response.codes.shape == (10, 3)
    assert b.status == "success" and b.response.action == "next"
    q.put(inf.GenerateRequest(request=dict(text="boom"), response_queue=rq))
    e = rq.get(timeout=10)
    assert e.status == "error" and isinstance(e.response, ValueError)
    q.put(None)  # shutdown sentinel


def _fake_dac():
    d = object.__new__(DAC)  # no GPU: bypass __init__, keep isinstance(x, DAC) true (vq_manager.py:19)
    d.sample_rate = 44100
    d._device = torch.device("cpu")
    d.from_indices = lambda codes: torch.full((codes.shape[0], 1, codes.shape[-1] * 2048), 0.25)
    return d


def _serve(q):
    while True:
        item = q.get()
        if item is None:
            return
        text = item.request["text"]
        if text == "fail":
            item.response_queue.put(inf.WrappedGenerateResponse(status="error", response=RuntimeError("lm died")))
            continue
        for _ in range(2):
            item.response_queue.put(inf.WrappedGenerateResponse(
                status="success", response=inf.GenerateResponse(action="sample", codes=torch.zeros(10, 2, dtype=torch.long))))
        item.response_queue.put(inf.WrappedGenerateResponse(status="success", response=inf.GenerateResponse(action="next")))


def test_tts_engine_streaming_and_errors():
    import threading

    q = queue.Queue()
    threading.Thread(target=_serve, args=(q,), daemon=True).start()
    eng = TTSInferenceEngine(q, _fake_dac(), torch.bfloat16, compile=False)
    res = list(eng.inference(ServeTTSRequest(text="hi", streaming=True, seed=3)))
    assert [r.code for r in res] == ["header", "segment", "segment", "final"]
    assert res[0].audio[0] == 44100 and res[-1].audio[1].shape == (2 * 2 * 2048,)
    assert res[-1].audio[1].dtype == np.float32 and np.allclose(res[-1].audio[1], 0.25)
    res = list(eng.inference(ServeTTSRequest(text="hi")))
    assert [r.code for r in res] == ["final"]
    res = list(eng.inference(ServeTTSRequest(text="fail")))
    assert res[0].code == "error" and isinstance(res[0].error, RuntimeError)
    q.put(None)


class _FakeStream:
    """Incremental decoder stand-in: sample value = absolute frame index, so ordering / completeness show in the audio."""

    def __init__(self):
        self.pos = 0

    def push(self, codes):
        k = codes.shape[-1]
        out = torch.arange(self.pos, self.pos + k, dtype=torch.float32).repeat_interleave(2048).view(1, 1, -1)
        self.pos += k
        return out


def test_tts_engine_streams_partial_codes():
    """Streaming request: the worker announces finished frames ("partial") while the chunk is still being generated;
    every piece is decoded incrementally and handed out at once, the chunk's "sample" only closes it (frames the worker
    did not announce are decoded then), a new chunk starts a new codec stream, and `final` is the concatenation."""
    import threading

    def serve(q):
        item = q.get()
        assert item.request["stream_frames"] == 8
        put = lambda a, n=0: item.response_queue.put(inf.WrappedGenerateResponse(
            status="success", response=inf.GenerateResponse(action=a, codes=torch.zeros(10, n, dtype=torch.long) if n else None)))
        put("partial", 8)
        put("partial", 5)
        put("sample", 15)   # 2 frames were never announced
        put("partial", 3)
        put("sample", 3)
        put("sample", 4)    # a chunk without partials: one-shot decode
        put("next")

    q = queue.Queue()
    threading.Thread(target=serve, args=(q,), daemon=True).start()
    dac = _fake_dac()
    dac.open_decode_stream = lambda batch=1, max_frames=4096: _FakeStream()
    eng = TTSInferenceEngine(q, dac, torch.bfloat16, compile=False)
    res = list(eng.inference(ServeTTSRequest(text="hi", streaming=True)))
    assert [r.code for r in res] == ["header"] + ["segment"] * 5 + ["final"]
    seg = [r.audio[1] for r in res[1:-1]]
    assert [len(x) // 2048 for x in seg] == [8, 5, 2, 3, 4]
    first_chunk = np.concatenate(seg[:3])
    assert np.array_equal(first_chunk[::2048], np.arange(15, dtype=np.float32))  # frames in order, none lost or repeated
    assert np.array_equal(seg[3][::2048], np.arange(3, dtype=np.float32))          # the next chunk restarts the stream
    assert np.allclose(seg[4], 0.25)                                               # one-shot from_indices
    assert np.array_equal(res[-1].audio[1], np.concatenate(seg))
    assert eng.last_first_audio_s is not None and eng.last_first_audio_s >= 0


def test_worker_forwards_partial_codes(monkeypatch):
    """launch_thread_safe_queue: `stream_frames` in a request makes the worker forward generate_long's on_partial
    calls as "partial" responses, in order, before the chunk's "sample"."""

    def fake_generate_long(*, model, decode_one_token, text, on_partial=None, **kw):
        assert "stream_frames" not in kw
        if on_partial is not None:
            on_partial(torch.ones(10, 8, dtype=torch.long))
            on_partial(torch.ones(10, 2, dtype=torch.long))
        yield inf.GenerateResponse(action="sample", codes=torch.ones(10, 10, dtype=torch.long), text=text)
        yield inf.GenerateResponse(action="next")

    monkeypatch.setattr(inf, "init_model", lambda *a, **k: (_FakeModel(), inf.decode_one_token_ar))
    monkeypatch.setattr(inf, "generate_long", fake_generate_long)
    q = inf.launch_thread_safe_queue("ckpt", "cpu", torch.bfloat16)
    rq = queue.Queue()
    q.put(inf.GenerateRequest(request=dict(text="hello", stream_frames=8), response_queue=rq))
    got = [rq.get(timeout=10) for _ in range(4)]
    assert [g.response.action for g in got] == ["partial", "partial", "sample", "next"]
    assert [g.response.codes.shape[-1] for g in got[:3]] == [8, 2, 10]
    q.put(inf.GenerateRequest(request=dict(text="plain"), response_queue=rq))
    got = [rq.get(timeout=10) for _ in range(2)]
    assert [g.response.action for g in got] == ["sample", "next"]
    q.put(None)


def test_wav_chunk_header_is_riff():
    from fish_speech_b200.inference_engine.utils import wav_chunk_header

    h = wav_chunk_header(44100)
    assert h[:4] == b"RIFF" and h[8:12] == b"WAVE"


def test_generate_long_validates_sampling_args():
    with pytest.raises(AssertionError):
        next(inf.generate_long(model=None, device="cpu", decode_one_token=None, text="x", top_p=0.0))
    with pytest.raises(AssertionError):
        next(inf.generate_long(model=None, device="cpu", decode_one_token=None, text="x", temperature=2.5))


class _FakeBatcher:
    """Stands in for scheduler.ContinuousBatcher: a request finishes after ceil(limit / 4) steps and its
    result is the prompt followed by `max_new_tokens` copies of its seed's low byte."""

    def __init__(self, slots):
        self.slots, self.waiting, self.active, self.max_active, self.closed = slots, [], [], 0, False

    def submit(self, r):
        self.waiting.append(r)

    def idle(self):
        return not self.waiting and not self.active

    def step(self):
        while self.waiting and len(self.active) < self.slots:
            r = self.waiting.pop(0)
            self.active.append([r, (r.max_new_tokens + 3) // 4])
        self.max_active = max(self.max_active, len(self.active))
        for e in list(self.active):
            e[1] -= 1
            if e[1] <= 0:
                self.active.remove(e)
                r = e[0]
                r.result = torch.cat([r.prompt, torch.full((r.prompt.size(0), r.max_new_tokens), 7)], dim=1)
                r.on_done(r)

    def close(self):
        self.closed = True


def _fake_plan(*, model, text, chunks=2, fail=False, **kw):
    """Shape of _generate_long_plan: per chunk one generate request, then a sample response; 'next' at the end."""
    for c in range(chunks):
        y = yield ("generate", dict(prompt=torch.full((3, 2 + c), len(text)), max_new_tokens=4 * (c + 1) + len(text),
                                    audio_masks=None, audio_parts=None, temperature=0.7, top_p=0.7, top_k=30))
        if fail:
            raise RuntimeError("boom")
        yield ("response", inf.GenerateResponse(action="sample", codes=y[1:, 2 + c:], text=f"{text}#{c}"))
    yield ("response", inf.GenerateResponse(action="next"))


def test_slot_scheduler_worker_interleaves_requests(monkeypatch):
    """serve_requests: several queued requests advance together, each response queue sees the reference's
    sequence (sample per chunk, then next), an exception reaches only its own request, None shuts down."""
    import queue as Q

    monkeypatch.setattr(inf, "_generate_long_plan", _fake_plan)
    fb = _FakeBatcher(slots=3)
    q = Q.Queue()
    outs = []
    for i, (text, fail) in enumerate([("a", False), ("bbbbbb", False), ("cc", True), ("ddd", False)]):
        rq = Q.Queue()
        outs.append(rq)
        q.put(inf.GenerateRequest(request=dict(text=text, fail=fail, chunks=2), response_queue=rq))
    q.put(None)
    inf.serve_requests(_FakeModel(), q, 3, batcher=fb)
    assert fb.closed and fb.max_active == 3  # three requests really shared the scheduler steps

    def drain(rq):
        items = []
        while not rq.empty():
            items.append(rq.get_nowait())
        return items

    for i, text in [(0, "a"), (1, "bbbbbb"), (3, "ddd")]:
        items = drain(outs[i])
        assert [it.status for it in items] == ["success"] * 3
        assert [it.response.action for it in items] == ["sample", "sample", "next"]
        assert [it.response.text for it in items[:2]] == [f"{text}#0", f"{text}#1"]
        assert items[0].response.codes.shape == (2, 4 + len(text))
        assert items[1].response.codes.shape == (2, 8 + len(text))
    bad = drain(outs[2])
    assert len(bad) == 1 and bad[0].status == "error" and isinstance(bad[0].response, RuntimeError)


def test_generate_long_drives_the_same_plan(monkeypatch):
    """generate_long = the plan driven one `generate` at a time (inference.py:611-721)."""
    monkeypatch.setattr(inf, "_generate_long_plan", _fake_plan)
    calls = []

    def fake_generate(*, model, prompt, max_new_tokens, seed, **kw):
        calls.append(seed)
        return torch.cat([prompt, torch.zeros(prompt.size(0), max_new_tokens, dtype=prompt.dtype)], dim=1)

    monkeypatch.setattr(inf, "generate", fake_generate)
    out = list(inf.generate_long(model=_FakeModel(), decode_one_token=None, text="xy", chunks=3))
    assert [r.action for r in out] == ["sample"] * 3 + ["next"]
    assert len(set(calls)) == 3  # every generate call gets its own Philox key


class _FakeEngine:
    """Host-visible behaviour of LmEngine under slot control, on CPU tensors: prefill writes the first frame of
    every admitted slot, a decode frame appends one token per live slot and freezes a slot at its limit."""

    def __init__(self, slots, kv_len=64, max_frames=32, max_rows=16):
        self.max_batch, self.kv_len, self.max_frames, self.max_rows = slots, kv_len, max_frames, max_rows
        self.device = torch.device("cpu")
        z = lambda *s, dt=torch.int32: torch.zeros(*s, dtype=dt)
        self.bufs = dict(slot_state=z(slots), slot_limit=z(slots), slot_temperature=z(slots, dt=torch.float32),
                         slot_top_p=z(slots, dt=torch.float32), slot_top_k=z(slots), slot_seed=z(slots, dt=torch.int64),
                         n_out=z(slots), pos=z(32), ras_window=z(slots, 10), out_tokens=z(slots, 3, max_frames))
        self.slot_control = False
        self.prefills, self.decodes, self.bounds = [], 0, []

    def buffer(self, name):
        return self.bufs[name]

    def reset(self):
        for k in ("slot_state", "n_out", "pos"):
            self.bufs[k].zero_()

    def set_slot_control(self, on):
        self.slot_control = bool(on)

    def set_context_bound_exact(self, n):
        self.bounds.append(n)

    def _frame(self, s):
        b = self.bufs
        if int(b["slot_state"][s]) != 1:
            return
        f = int(b["n_out"][s])
        b["out_tokens"][s, :, f] = 100 * s + f
        b["n_out"][s] = f + 1
        if f + 1 >= int(b["slot_limit"][s]):
            b["slot_state"][s] = 2
        else:
            b["pos"][s] += 1

    def prefill(self, prompts, slots, sp, start_pos=None, do_sample=True):
        assert sp is None and self.slot_control
        self.prefills.append(list(slots))
        for p, s in zip(prompts, slots):
            self.bufs["pos"][s] = p.shape[1]
            self._frame(s)

    def decode(self, batch, nframes, sp, use_graph=True):
        assert sp is None and batch == self.max_batch
        self.decodes += nframes
        for _ in range(nframes):
            for s in range(batch):
                self._frame(s)


class _SchedModel:
    def __init__(self, eng, max_seq_len=64):
        self.engine, self.max_batch_size = eng, eng.max_batch
        self.config = type("C", (), dict(max_seq_len=max_seq_len, num_codebooks=2))()


def test_continuous_batcher_host_logic():
    """scheduler.ContinuousBatcher against a fake engine: budgets (generate's max_new_tokens clamp, inference.py:
    270-279), slot reuse, grouped admissions, retirement order, engine handed back on close."""
    from fish_speech_b200.scheduler import ContinuousBatcher, SlotRequest

    eng = _FakeEngine(slots=2)
    model = _SchedModel(eng)
    b = ContinuousBatcher(model, max_slots=2, frames_per_poll=4)
    assert eng.slot_control
    order = []
    mk = lambda T, n, tag: SlotRequest(prompt=torch.full((3, T), tag), max_new_tokens=n, tag=tag,
                                       on_done=lambda r: order.append(r.tag))
    reqs = [b.submit(mk(5, 3, 0)), b.submit(mk(7, 9, 1)), b.submit(mk(4, 1, 2)), b.submit(mk(6, 0, 3))]
    assert reqs[3]._limit == min(64 - 6, eng.max_frames)  # max_new_tokens=0 -> as many as fit
    with pytest.raises(ValueError):
        b.submit(mk(64, 4, 9))  # prompt as long as max_seq_len (inference.py:262-265)
    b.run()
    assert b.idle() and sorted(order) == [0, 1, 2, 3] and order[0] == 0  # the 3-frame request leaves first
    assert eng.prefills[0] == [0, 1] and all(len(p) <= 2 for p in eng.prefills)  # two slots, reused afterwards
    assert sum(len(p) for p in eng.prefills) == 4
    for r, n in zip(reqs, [3, 9, 1, reqs[3]._limit]):
        T = r.prompt.size(1)
        assert r.result.shape == (3, T + n) and torch.equal(r.result[:, :T], r.prompt)
        assert r.result[0, T:].tolist() == [100 * r.slot + f for f in range(n)]  # its own frames, in order
    assert 0 < b.slot_frames <= b.frames_run * 2 and max(eng.bounds) <= eng.kv_len + 1
    b.close()
    assert not eng.slot_control and int(eng.bufs["slot_state"].sum()) == 0

    # grouped admissions: with min_free_to_admit=2 a single freed slot waits for the second one
    eng2 = _FakeEngine(slots=2)
    b2 = ContinuousBatcher(_SchedModel(eng2), max_slots=2, frames_per_poll=2, min_free_to_admit=2)
    for tag, n in enumerate([2, 8, 4, 4]):
        b2.submit(mk(3, n, tag))
    b2.run()
    assert eng2.prefills == [[0, 1], [0, 1]]  # the short request's slot was not refilled on its own


class _FakeCodec:
    """encode() of a DAC: codes[b, c, t] = c + 10 * (sample count of clip b) for t < ceil(len / hop)."""
    sample_rate, hop = 100, 10
    device = torch.device("cpu")

    def __init__(self):
        self.batches = []

    def encode(self, audios, lengths):
        B, _, N = audios.shape
        self.batches.append((B, N, lengths.tolist()))
        T = -(-N // self.hop)
        codes = torch.arange(3).view(1, 3, 1).expand(B, 3, T) + 10 * lengths.view(B, 1, 1)
        return codes.to(torch.int64), -(-lengths // self.hop)


def _write_wav(path, n, sr=100, nch=1):
    import wave

    with wave.open(str(path), "wb") as f:
        f.setnchannels(nch)
        f.setsampwidth(2)
        f.setframerate(sr)
        f.writeframes((np.arange(n * nch) % 100).astype("<i2").tobytes())


def test_bulk_encode_pipeline(tmp_path, monkeypatch):
    """fish_speech_b200/bulk_encode.py (the job of tools/vqgan/extract_vq.py): shard stride, skip of finished files,
    length-grouped padded batches, per-file trimming of the codes, unreadable files skipped, stereo down-mix."""
    from fish_speech_b200 import bulk_encode as be

    lens = [95, 12, 40, 41, 230, 13, 39, 11]
    for i, n in enumerate(lens):
        _write_wav(tmp_path / f"a{i}.wav", n, nch=2 if i == 2 else 1)
    (tmp_path / "broken.wav").write_bytes(b"not a wav")
    (tmp_path / "notes.txt").write_text("x")
    np.save(tmp_path / "a1.npy", np.zeros((3, 2)))  # already done -> skipped
    files = be.list_audio_files(tmp_path)
    assert [f.name for f in files] == sorted([f"a{i}.wav" for i in range(8)] + ["broken.wav"])

    monkeypatch.setenv("SLURM_PROCID", "1")
    monkeypatch.setenv("SLURM_NTASKS", "2")
    assert be.worker_identity() == (1, 2)
    todo_all = be.pending_files(files, 0, 1)
    assert tmp_path / "a1.wav" not in todo_all and len(todo_all) == 8
    assert be.pending_files(files, 1, 2) == todo_all[1::2]

    # batch planning: similar lengths share a batch, caps respected, every index exactly once
    plan = be.plan_batches([95, 40, 41, 230, 13, 39, 11], batch_size=3, max_padded_samples=300)
    assert sorted(i for b in plan for i in b) == list(range(7))
    assert all(len(b) <= 3 for b in plan) and [3] in plan  # the 230-sample clip cannot share a 300-sample budget
    assert any(set(b) == {1, 2, 5} or set(b) >= {1, 2} for b in plan)

    codec = _FakeCodec()
    n, secs = be.encode_files(todo_all, codec, batch_size=3, max_batch_seconds=3.0)
    assert n == 7 and abs(secs - sum(lens[i] for i in (0, 2, 3, 4, 5, 6, 7)) / 100) < 1e-6  # broken.wav skipped
    for i in (0, 2, 3, 4, 5, 6, 7):
        got = np.load(tmp_path / f"a{i}.npy")
        assert got.shape == (3, -(-lens[i] // 10)) and got.dtype == np.int64
        assert (got[:, 0] == np.arange(3) + 10 * lens[i]).all()  # its own codes, trimmed to its own length
    assert np.load(tmp_path / "a1.npy").shape == (3, 2)  # untouched
    assert not (tmp_path / "broken.npy").exists() and not list(tmp_path.glob("*.tmp"))
    assert all(B <= 3 and B * N <= 300 for B, N, _ in codec.batches)
    # everything is done now: a second pass finds nothing
    assert be.pending_files(be.list_audio_files(tmp_path), 0, 1) == [tmp_path / "broken.wav"]


def test_extract_vq_spawn_plan():
    import importlib.util
    from pathlib import Path

    spec = importlib.util.spec_from_file_location("extract_vq", Path(__file__).resolve().parent.parent / "tools/vqgan/extract_vq.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    plan = mod.spawn_plan(4, ["0", "3"])
    assert [p["CUDA_VISIBLE_DEVICES"] for p in plan] == ["0", "3", "0", "3"]
    assert [p["SLURM_PROCID"] for p in plan] == ["0", "1", "2", "3"] and {p["SLURM_NTASKS"] for p in plan} == {"4"}


def test_slot_scheduler_worker_reports_engine_failure(monkeypatch):
    """If the batcher itself fails (a CUDA error, say) every request in flight receives an error response, and so
    does every request that arrives afterwards: the worker keeps answering instead of dying with callers blocked on
    their queues (the reference's worker catches per request and keeps serving, inference.py:748-799). `None` ends it;
    a close() that fails on the broken engine does not mask anything."""
    import queue as Q
    import threading

    monkeypatch.setattr(inf, "_generate_long_plan", _fake_plan)

    class Boom(_FakeBatcher):
        def step(self):
            raise RuntimeError("device lost")

        def close(self):
            self.closed = True
            raise RuntimeError("reset failed too")

    fb = Boom(slots=2)
    q, outs = Q.Queue(), [Q.Queue(), Q.Queue()]
    for rq in outs:
        q.put(inf.GenerateRequest(request=dict(text="ab", chunks=1), response_queue=rq))
    t = threading.Thread(target=inf.serve_requests, args=(_FakeModel(), q, 2), kwargs=dict(batcher=fb), daemon=True)
    t.start()
    for rq in outs:
        item = rq.get(timeout=20)
        assert item.status == "error" and "device lost" in str(item.response)
    late = Q.Queue()
    q.put(inf.GenerateRequest(request=dict(text="late", chunks=1), response_queue=late))
    item = late.get(timeout=20)
    assert item.status == "error" and "device lost" in str(item.response)
    q.put(None)
    t.join(timeout=20)
    assert not t.is_alive() and fb.closed


def test_continuous_batcher_rejects_bad_requests_up_front():
    """Per-request errors surface in submit() (so the worker can answer that request alone), not in the engine."""
    from fish_speech_b200.scheduler import ContinuousBatcher, SlotRequest

    b = ContinuousBatcher(_SchedModel(_FakeEngine(slots=2)), max_slots=2)
    ok = dict(prompt=torch.zeros(3, 4, dtype=torch.long), max_new_tokens=4)
    for bad in (dict(top_k=0), dict(top_p=0.0), dict(top_p=1.5), dict(temperature=0.0), dict(temperature=2.0),
                dict(prompt=torch.zeros(2, 4, dtype=torch.long)), dict(prompt=torch.zeros(3, 4)),
                dict(prompt=torch.zeros(3, 0, dtype=torch.long))):
        with pytest.raises(ValueError):
            b.submit(SlotRequest(**{**ok, **bad}))
    b.submit(SlotRequest(**ok))
    assert len(b.waiting) == 1


class _ByteTokenizer:
    """Stand-in for FishTokenizer (fish_speech/tokenizer.py): bytes are ids 0..255, the handful of special tokens the
    prompt builder emits get ids from 256, semantic tokens start at 1000."""

    semantic_begin_id, semantic_end_id = 1000, 1000 + 4095

    def __init__(self):
        import re

        self.special = {}
        self._re = re.compile(r"(<\|[^|]+\|>)")

    def get_token_id(self, token):
        return self.special.setdefault(token, 256 + len(self.special))

    def encode(self, text, add_special_tokens=False, **kw):
        ids = []
        for piece in self._re.split(text):
            if not piece:
                continue
            ids += [self.get_token_id(piece)] if self._re.fullmatch(piece) else list(piece.encode("utf-8"))
        return ids


FRONTEND_GOLD = Path(__file__).parent / "golden" / "generate_long_frontend.npz"


def _frontend_value(v):
    """JSON form of an argument the generate_long plan passes to the prompt builder (nested parts and tensors included)."""
    if isinstance(v, torch.Tensor):
        return {"dtype": str(v.dtype), "shape": list(v.shape), "values": v.flatten().tolist()}
    if isinstance(v, (list, tuple)):
        return [_frontend_value(x) for x in v]
    if hasattr(v, "frontend_call"):
        kind, kw = v.frontend_call
        return {"kind": kind, **{k: _frontend_value(x) for k, x in kw.items()}}
    return v


def frontend_conversation_json(messages) -> str:
    """Every Message of a conversation as the plan constructed it (constructor, keyword arguments, parts)."""
    return json.dumps([_frontend_value(m) for m in messages], sort_keys=True)


def _recorded_frontend(gold):
    """Stand-in for the reference's prompt builder (fish_speech.conversation / content_sequence) that replays a recorded
    run of the real one (oracle/make_golden_frontend.py): the k-th encode_for_inference must be asked to encode exactly
    the conversation the reference encoded k-th, and returns the reference's prompt for it."""
    calls = iter(range(len(gold["conversations"])))

    class Call:
        def __init__(self, kind, **kw):
            self.frontend_call = (kind, kw)

    class Conversation:
        def __init__(self):
            self.messages = []

        def append(self, message):
            self.messages.append(message)

        def encode_for_inference(self, tokenizer, num_codebooks):
            k = next(calls, None)
            assert k is not None, "the plan encodes more prompts than the recorded reference run"
            assert num_codebooks == int(gold["num_codebooks"])
            assert frontend_conversation_json(self.messages) == str(gold["conversations"][k]), \
                f"prompt {k}: the plan built a different conversation than the recorded reference run"
            return torch.from_numpy(gold[f"encoded_{k}"]), None, None

    def part(kind):
        return lambda **kw: Call(kind, **kw)

    return part("TextPart"), part("VQPart"), Conversation, part("Message")


def drive_generate_long_plan(tok):
    """The REAL body of the generate_long plan (inference.py:523-733) with a byte-level tokenizer and a driver that
    answers every `generate` with a made-up continuation. Returns (prompts, responses, reference clip codes)."""

    class Model:
        class config:
            max_seq_len, num_codebooks = 8192, 10

        tokenizer = tok

    ref_codes = torch.arange(10 * 6).view(10, 6) % 1024
    text = "<|speaker:0|>" + "first sentence of the request. " * 3 + "<|speaker:1|>" + "and a reply that is long enough. " * 3
    plan = inf._generate_long_plan(model=Model, device="cpu", text=text, chunk_length=100, max_new_tokens=64,
                                   temperature=0.8, top_p=0.8, top_k=30, prompt_text=["reference words"],
                                   prompt_tokens=[ref_codes])
    prompts, responses, reply, fake_frames = [], [], None, 0
    while True:
        try:
            kind, payload = plan.send(reply)
        except StopIteration:
            break
        reply = None
        if kind == "response":
            responses.append(payload)
            continue
        p = payload["prompt"]
        assert payload["reuse_prefix"] is True and payload["max_new_tokens"] == 64
        assert p.shape[0] == 11 and p.dtype in (torch.int32, torch.int64)
        prompts.append(p.clone())
        fake_frames += 1
        n = 4 + fake_frames  # frames this "generate" produced; the last one is <|im_end|>
        gen = torch.zeros(11, n, dtype=p.dtype)
        gen[0] = tok.semantic_begin_id + 7 * fake_frames
        gen[1:] = (torch.arange(10).view(10, 1) + fake_frames) % 1024
        gen[0, -1] = tok.get_token_id("<|im_end|>")
        reply = torch.cat([p, gen], dim=1)
    return prompts, responses, ref_codes


def test_generate_long_plan_builds_growing_prompts_with_the_reference_frontend(monkeypatch):
    """The generate_long plan against a recorded run of the reference's own prompt builder (fish_speech.content_sequence /
    conversation, tests/golden/generate_long_frontend.npz): the plan must hand the builder the same conversations, chunk
    by chunk. Checks on the reference's prompts what the CUDA side relies on: every chunk's prompt EXTENDS the previous
    chunk's prompt (prefix K/V reuse, SURVEY §8(f).2), the reference clip enters as semantic rows, each chunk yields
    y[1:, T:-1] (the last frame is dropped, :708) and the stream ends with "next"."""
    gold = np.load(FRONTEND_GOLD)
    monkeypatch.setattr(inf, "_reference_frontend", lambda: _recorded_frontend(gold))
    tok = _ByteTokenizer()
    tok.special = json.loads(str(gold["tokenizer_special"]))
    prompts, responses, ref_codes = drive_generate_long_plan(tok)
    assert len(prompts) == len(gold["conversations"])
    assert len(prompts) >= 2, "the text must split into several chunks"
    # the reference clip: semantic ids on row 0, its codes on rows 1..10
    first = prompts[0]
    sem = (first[0] >= tok.semantic_begin_id) & (first[0] <= tok.semantic_end_id)
    assert int(sem.sum()) == 6 and torch.equal(first[1:, sem], ref_codes.to(first.dtype))
    assert torch.equal(first[0, sem], (ref_codes[0] + tok.semantic_begin_id).to(first.dtype))
    assert int(first[1:, ~sem].abs().sum()) == 0  # text rows carry no codes
    for a, b in zip(prompts, prompts[1:]):
        assert b.shape[1] > a.shape[1] and torch.equal(b[:, : a.shape[1]], a), "a chunk's prompt must extend the previous one"
    # previous generations come back as semantic rows right after the previous prompt
    k = prompts[0].shape[1]
    assert torch.equal(prompts[1][1:, k: k + 4], ((torch.arange(10).view(10, 1) + 1) % 1024).expand(10, 4).to(prompts[1].dtype))
    kinds = [r.action for r in responses]
    assert kinds == ["sample"] * len(prompts) + ["next"]
    for i, r in enumerate(responses[:-1]):
        assert r.codes.shape == (10, 4 + i) and torch.equal(r.codes[:, 0], (torch.arange(10) + i + 1) % 1024)


def test_continuous_batcher_streams_final_frames_per_request():
    """SlotRequest.on_frames (SURVEY 8f.3 in the slot scheduler): after every poll a streaming request receives the codes
    of the frames that are final -- all but its newest -- and over its lifetime exactly result[1:, T:-1], before on_done;
    requests without the callback are untouched; two requests of different lengths stream independently."""
    from fish_speech_b200.scheduler import ContinuousBatcher, SlotRequest

    eng = _FakeEngine(slots=2, max_frames=32)
    b = ContinuousBatcher(_SchedModel(eng), max_slots=2, frames_per_poll=4)
    got = {0: [], 1: []}
    order = []
    mk = lambda i, n, stream: SlotRequest(
        prompt=torch.full((3, 5), i, dtype=torch.long), max_new_tokens=n, tag=i,
        on_frames=(lambda r, codes: (got[r.tag].append(codes.clone()), order.append(("frames", r.tag)))) if stream else None,
        on_done=lambda r: order.append(("done", r.tag)))
    r0, r1, r2 = mk(0, 11, True), mk(1, 6, True), mk(2, 7, False)
    for r in (r0, r1, r2):
        b.submit(r)
    b.run()
    for r in (r0, r1):
        kept = r.result[1:, 5:-1]
        cat = torch.cat(got[r.tag], dim=1)
        assert torch.equal(cat.to(kept.dtype), kept), (r.tag, cat.shape, kept.shape)
        assert len(got[r.tag]) >= 2 and all(c.device.type == "cpu" for c in got[r.tag])
        assert order.index(("done", r.tag)) > max(i for i, e in enumerate(order) if e == ("frames", r.tag))
    assert r2.result.shape[1] == 5 + 7 and ("frames", 2) not in order


def test_slot_scheduler_worker_sends_partials_for_streaming_requests(monkeypatch):
    """serve_requests with `stream_frames` in a request: "partial" responses (codes of final frames) arrive on that
    request's queue ahead of each chunk's "sample" and add up to the sample's codes; other requests see none."""
    import queue as Q

    from fish_speech_b200.scheduler import ContinuousBatcher

    def plan(*, model, text, **kw):
        for c in range(2):
            y = yield ("generate", dict(prompt=torch.full((3, 4), 1, dtype=torch.long), max_new_tokens=9 + c, audio_masks=None,
                                        audio_parts=None, temperature=0.7, top_p=0.7, top_k=30))
            yield ("response", inf.GenerateResponse(action="sample", codes=y[1:, 4:-1], text=f"{text}#{c}"))
        yield ("response", inf.GenerateResponse(action="next"))

    monkeypatch.setattr(inf, "_generate_long_plan", plan)
    eng = _FakeEngine(slots=2, max_frames=32)
    model = _SchedModel(eng)
    model._philox_calls = 0
    b = ContinuousBatcher(model, max_slots=2, frames_per_poll=4)
    q, rs, rn = Q.Queue(), Q.Queue(), Q.Queue()
    q.put(inf.GenerateRequest(request=dict(text="s", stream_frames=8), response_queue=rs))
    q.put(inf.GenerateRequest(request=dict(text="n"), response_queue=rn))
    q.put(None)
    inf.serve_requests(model, q, 2, batcher=b)
    items = []
    while not rs.empty():
        items.append(rs.get_nowait())
    assert all(it.status == "success" for it in items)
    acts = [it.response.action for it in items]
    assert acts[-1] == "next" and acts.count("sample") == 2 and acts.count("partial") >= 2
    i0 = acts.index("sample")
    first = torch.cat([it.response.codes for it in items[:i0]], dim=1)
    assert set(acts[:i0]) == {"partial"} and torch.equal(first.to(items[i0].response.codes.dtype), items[i0].response.codes)
    i1 = acts.index("sample", i0 + 1)
    second = torch.cat([it.response.codes for it in items[i0 + 1:i1]], dim=1)
    assert torch.equal(second.to(items[i1].response.codes.dtype), items[i1].response.codes)
    plain = []
    while not rn.empty():
        plain.append(rn.get_nowait().response.action)
    assert plain == ["sample", "sample", "next"]


def test_batch_encode_pads_once_and_cuts_each_item(tmp_path):
    """bulk_encode.batch_encode (tools/server/model_utils.py:15-48): encoded bytes and waveforms mixed, ONE padded
    encode call, per-item codes cut to that item's frames."""
    from fish_speech_b200 import bulk_encode as BE

    codec = _FakeCodec()
    f = tmp_path / "a.wav"
    _write_wav(f, 57, sr=100)
    items = [f.read_bytes(), torch.zeros(1, 31), torch.zeros(1, 90)]
    outs = BE.batch_encode(codec, items)
    assert codec.batches == [(3, 90, [57, 31, 90])]
    assert [tuple(o.shape) for o in outs] == [(3, 6), (3, 4), (3, 9)]
    assert int(outs[0][1, 0]) == 1 + 570 and int(outs[2][2, -1]) == 2 + 900
    assert BE.batch_encode(codec, []) == []


def test_reference_loader_caches_by_hash_and_by_id(tmp_path, monkeypatch):
    """ReferenceLoader (reference_loader.py:62-160): one encode per distinct uploaded audio unless the request turns the
    cache off; library ids are validated and read clip + .lab pairs; load_audio decodes bytes and paths to mono float32."""
    from fish_speech_b200.inference_engine import reference_loader as RL

    monkeypatch.setattr(RL, "LIBRARY", tmp_path / "references")
    calls = []

    class L(RL.ReferenceLoader):
        def encode_reference(self, reference_audio, enable_reference_audio):
            calls.append(len(reference_audio))
            return torch.full((2, 3), len(reference_audio))

    ld = L()
    R = lambda a, t: type("Ref", (), dict(audio=a, text=t))()
    refs = [R(b"aaaa", "one"), R(b"bb", "two"), R(b"aaaa", "one again")]
    toks, texts = ld.load_by_hash(refs, "on")
    assert calls == [4, 2] and texts == ["one", "two", "one"] and int(toks[2][0, 0]) == 4
    ld.load_by_hash(refs[:1], "on")
    assert calls == [4, 2]
    ld.load_by_hash(refs[:1], "off")
    assert calls == [4, 2, 4]
    with pytest.raises(ValueError):
        ld.load_by_id("../etc", "on")
    d = tmp_path / "references" / "voice 1"
    d.mkdir(parents=True)
    _write_wav(d / "a.wav", 50, sr=100)
    (d / "a.lab").write_text("hello", encoding="utf-8")
    (d / "notes.txt").write_text("x")
    toks, texts = ld.load_by_id("voice 1", "on")
    assert texts == ["hello"] and len(toks) == 1 and ld.list_reference_ids() == ["voice 1"]
    n = len(calls)
    ld.load_by_id("voice 1", "on")
    assert len(calls) == n
    wav = ld.load_audio((d / "a.wav").read_bytes(), 100)
    assert wav.dtype == np.float32 and wav.shape == (50,)
    assert np.array_equal(ld.load_audio(str(d / "a.wav"), 100), wav)


def test_wav_chunk_header_is_the_header_of_an_empty_pcm_wav():
    import io
    import wave

    from fish_speech_b200.inference_engine.utils import pcm16, wav_chunk_header

    for sr, bits, ch in ((44100, 16, 1), (16000, 16, 2), (48000, 32, 1)):
        buf = io.BytesIO()
        with wave.open(buf, "wb") as f:
            f.setnchannels(ch)
            f.setsampwidth(bits // 8)
            f.setframerate(sr)
        assert wav_chunk_header(sr, bits, ch) == buf.getvalue()
    assert pcm16(np.array([0.0, 1.0, -1.0, 2.0, 0.5])) == np.array([0, 32767, -32767, 32767, 16383], dtype="<i2").tobytes()
