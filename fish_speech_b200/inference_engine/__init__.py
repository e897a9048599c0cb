"""TTSInferenceEngine — the surface of fish_speech/inference_engine/__init__.py (`inference` :22-142,
`send_Llama_request` :144-177, `get_audio_segment` :179-192) with the codec stage overlapped with generation.

The reference turns a chunk's codes into audio only after the LM has finished the chunk. Here a streaming request asks
the LM worker for the codes of finished frames while it keeps decoding (`stream_frames`, "partial" responses), and this
thread pushes them through an incremental codec decoder (`DAC.open_decode_stream`) on its own CUDA stream: audio leaves
with a delay of a few frames instead of a whole chunk (SURVEY §8(f).3). Non-streaming requests follow the reference:
one `from_indices` per chunk. The result protocol is the reference's: header | segment* | final, or error.
"""
from __future__ import annotations

import os
import queue
import time
from typing import Generator, Optional

import numpy as np
import torch

from ..models.dac.modded_dac import DAC
from ..models.text2semantic.inference import GenerateRequest, GenerateResponse, WrappedGenerateResponse
from .reference_loader import ReferenceLoader
from .schema import ServeTTSRequest
from .utils import InferenceResult, wav_chunk_header
from .vq_manager import VQManager

try:
    from loguru import logger
except Exception:  # pragma: no cover
    import logging

    logger = logging.getLogger("fish_speech_b200")


def set_seed(seed: int):
    """fish_speech/utils/utils.py:120-134: one seed for every generator the request may touch."""
    import random

    seed = min(abs(int(seed)), 1 << 31)
    random.seed(seed)
    np.random.seed(seed)
    torch.manual_seed(seed)
    if torch.cuda.is_available():
        torch.cuda.manual_seed_all(seed)


class _ChunkAudio:
    """Audio of the text chunk being generated: filled piece by piece (streaming) or in one go."""

    def __init__(self, engine: "TTSInferenceEngine"):
        self.engine = engine
        self.stream = None
        self.pieces: list[np.ndarray] = []
        self.frames = 0

    def push_partial(self, codes: torch.Tensor) -> np.ndarray:
        if self.stream is None:
            self.stream = self.engine.open_decode_stream()
        wav = self.stream.push(codes[None])[0, 0].float().cpu().numpy()
        self.pieces.append(wav)
        self.frames += codes.shape[-1]
        return wav

    def finish(self, codes: torch.Tensor) -> Optional[np.ndarray]:
        """End of the chunk: `codes` are all of its frames. Returns audio that has not been handed out yet."""
        rest = None
        if self.frames == 0:  # nothing was streamed: the reference's one-shot decode
            rest = self.engine.decode_vq_tokens(codes=codes).float().cpu().numpy()
            self.pieces.append(rest)
        elif self.frames < codes.shape[-1]:  # frames the worker did not announce separately
            rest = self.push_partial(codes[:, self.frames:])
        return rest

    def audio(self) -> np.ndarray:
        return np.concatenate(self.pieces, axis=0)


class TTSInferenceEngine(ReferenceLoader, VQManager):
    def __init__(self, llama_queue: queue.Queue, decoder_model: DAC, precision: torch.dtype, compile: bool) -> None:
        super().__init__()
        self.llama_queue = llama_queue
        self.decoder_model = decoder_model
        self.precision = precision
        self.compile = compile
        self.stream_frames = int(os.environ.get("FSB_STREAM_FRAMES", "8"))
        self.last_first_audio_s: Optional[float] = None  # request start -> first audio samples handed out

    @torch.inference_mode()
    def inference(self, req: ServeTTSRequest) -> Generator[InferenceResult, None, None]:
        t_start = time.perf_counter()
        self.last_first_audio_s = None
        if req.reference_id is not None:
            prompt_tokens, prompt_texts = self.load_by_id(req.reference_id, req.use_memory_cache)
        elif req.references:
            prompt_tokens, prompt_texts = self.load_by_hash(req.references, req.use_memory_cache)
        else:
            prompt_tokens, prompt_texts = [], []
        if req.seed is not None:
            set_seed(req.seed)
            logger.warning(f"set seed: {req.seed}")
        responses = self.send_Llama_request(req, prompt_tokens, prompt_texts)
        rate = self.decoder_model.sample_rate
        if req.streaming:
            yield InferenceResult(code="header", audio=(rate, np.array(wav_chunk_header(sample_rate=rate))), error=None)
        finished: list[np.ndarray] = []
        chunk = _ChunkAudio(self)

        def hand_out(wav):
            if self.last_first_audio_s is None:
                self.last_first_audio_s = time.perf_counter() - t_start
            return InferenceResult(code="segment", audio=(rate, wav), error=None)

        # a CUDA stream of our own: the LM worker thread keeps its stream busy with decode frames meanwhile
        dev = torch.device(self.decoder_model.device)
        side = torch.cuda.Stream(device=dev) if dev.type == "cuda" else None
        while True:
            wrapped: WrappedGenerateResponse = responses.get()
            if wrapped.status == "error":
                err = wrapped.response if isinstance(wrapped.response, Exception) else Exception("Unknown error")
                yield InferenceResult(code="error", audio=None, error=err)
                return
            result = wrapped.response
            if not isinstance(result, GenerateResponse):
                raise TypeError(f"Expected GenerateResponse, got {type(result).__name__}")
            if result.action == "next":
                break
            with (torch.cuda.stream(side) if side is not None else _nullcontext()):
                if result.action == "partial":
                    wav = chunk.push_partial(result.codes)
                else:  # "sample": the chunk is complete
                    wav = chunk.finish(result.codes)
                    finished.append(chunk.audio())
                    chunk = _ChunkAudio(self)
            if wav is not None and wav.size and req.streaming:
                yield hand_out(wav)
        if not finished:
            yield InferenceResult(code="error", audio=None,
                                  error=RuntimeError("No audio generated, please check the input text."))
            return
        if self.last_first_audio_s is None:
            self.last_first_audio_s = time.perf_counter() - t_start
        yield InferenceResult(code="final", audio=(rate, np.concatenate(finished, axis=0)), error=None)

    def send_Llama_request(self, req: ServeTTSRequest, prompt_tokens: list, prompt_texts: list) -> queue.Queue:
        """Queue one generate_long call on the LM worker (inference.py:736-799); the answer comes on the returned queue."""
        request = dict(
            device=self.decoder_model.device, max_new_tokens=req.max_new_tokens, text=req.text, top_p=req.top_p,
            repetition_penalty=req.repetition_penalty, temperature=req.temperature, compile=self.compile,
            iterative_prompt=req.chunk_length > 0, chunk_length=req.chunk_length, prompt_tokens=prompt_tokens,
            prompt_text=prompt_texts)
        if req.streaming and self.stream_frames > 0:
            request["stream_frames"] = self.stream_frames
        response_queue: queue.Queue = queue.Queue()
        self.llama_queue.put(GenerateRequest(request=request, response_queue=response_queue))
        return response_queue

    def get_audio_segment(self, result: GenerateResponse) -> np.ndarray:
        """One-shot decode of a finished chunk. The codec computes in bf16 with fp32 accumulation whatever `precision`
        says (the reference wraps this call in torch.autocast(bf16), inference_engine/__init__.py:185-189)."""
        return self.decode_vq_tokens(codes=result.codes).float().cpu().numpy()


class _nullcontext:
    def __enter__(self):
        return None

    def __exit__(self, *a):
        return False
