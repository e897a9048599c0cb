#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native Fish-Speech hot path.

Workload (BASELINE.json configs[2]): batch-32 text->codec->wav, 64-token prompts, 256 codec frames per
utterance, bf16, greedy (top_k=1), synthetic seeded weights at the assumed S2-Pro geometry
(SURVEY.md §8) — one "step" = the whole batch: prefill + 255 decode frames (+ codec decode to waveform
once the codec stage is present in this build; `config.stages` says which stages were timed).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Prints ONE JSON line.  `value` = audio-seconds generated per second (whole job, all GPUs) with the prompts
resident in HBM; `e2e` = the same through the public API (`generate_batch`) from pinned host memory,
including H2D of the prompts and D2H of the generated codes; `roofline` = measured HBM stream of the
dominant kernel (the tcgen05 weight-streaming step GEMM) against MEASURED_PEAKS.json, in the frame and as a
GEMM-only replay; `cpu_baseline` = the reference's CPU path (oracle/cpu_baseline.py) timed on this box's host
cores on a bounded sample.

Under torchrun (N > 1) every rank runs a full replica on its own shard of utterances (32 per GPU, weak
scaling, no collective on the data path); times are device-side, max over ranks.

`--dump-outputs DIR` (batch32, one GPU) also writes what the last timed step computed as DIR/<name>.npy (see
dump_outputs). Prompts and weights are seeded, the same on every run, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

SR, FRAME = 44100, 2048
B_PER_GPU, T_PROMPT, N_FRAMES = 32, 64, 256


def s2pro_cfg():
    from fish_speech_b200.configs import s2pro_args

    return s2pro_args(max_seq_len=512)


def codec_decode_macs(c, T: int) -> float:
    """Multiply-accumulates of DAC.from_indices for one utterance of T frames (every conv / linear /
    attention product; SURVEY §8: 866.9 GMAC at T=256 for the full geometry)."""
    D = c.latent_dim
    t = c.quant_tfm
    macs = 0.0
    per_tok = t.n_layer * (3 * t.dim * t.n_head * t.head_dim + t.dim * t.n_head * t.head_dim + 3 * t.dim * t.intermediate_size)
    win = t.window_size or T
    attn = t.n_layer * 2 * t.n_head * t.head_dim * sum(min(i + 1, win) for i in range(T))
    macs += per_tok * T + attn
    Tc = T
    for f in reversed(c.downsample_factor):
        macs += Tc * D * D * f  # transposed conv k = stride = f
        Tc *= f
        macs += Tc * (7 * D + 2 * 4 * D * D)  # ConvNeXt: depthwise k7 + two pointwise
    macs += Tc * 7 * D * c.decoder_dim
    cin = c.decoder_dim
    for s_ in c.decoder_rates:
        cout = cin // 2
        macs += Tc * cin * cout * 2 * s_  # transposed conv k = 2*stride: 2 taps per output phase, s phases
        Tc *= s_
        macs += 3 * Tc * (7 * cout * cout + cout * cout)
        cin = cout
    macs += Tc * 7 * cin
    return macs


def make_prompts(cfg, n, first_seed):
    """SURVEY §8(d) config 2/3: row 0 = random text ids, rows 1..10 = 0; seeds 42, 43, ..."""
    out = []
    for i in range(n):
        g = torch.Generator().manual_seed(first_seed + i)
        p = torch.zeros(cfg.num_codebooks + 1, T_PROMPT, dtype=torch.int32)
        p[0] = torch.randint(0, 151643, (T_PROMPT,), generator=g, dtype=torch.int32)
        out.append(p)
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.p = index, [], None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.p:
            self.p.terminate()
        sm = sorted(int(r[1]) for r in self.rows if len(r) > 2 and r[1].isdigit())
        mx = [int(r[2]) for r in self.rows if len(r) > 2 and r[2].isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.strip().lower() == "active":
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed
    `ncu --set full` capture (profiles/r02_step_gemm_ncu_full.json); None if no capture is committed."""
    try:
        d = json.loads((ROOT / "profiles" / "r02_step_gemm_ncu_full.json").read_text())
        return d["avg_dram_bytes_per_launch"]
    except Exception:
        return None


def peaks():
    try:
        return json.loads((ROOT / "MEASURED_PEAKS.json").read_text()), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def cpu_reference(steps: int, warmup: int):
    """The reference's own CPU implementation of the path on this box's host cores (oracle/cpu_baseline.py:
    the unmodified reference modules when /root/reference exists, else the pinned oracle port)."""
    from oracle import cpu_baseline

    return cpu_baseline.measure(steps, warmup)


DUMP_WAV_SAMPLES = 1 << 21  # 8 MiB of float32 (+ 16 MiB of float64 indices): the whole batch's waveform is 64 MiB


def dump_outputs(out_dir: Path, codes: torch.Tensor, wav: torch.Tensor | None) -> None:
    """What a caller of the timed path receives: `codes.npy` = the generated frames [B, C+1, NF] in float32 (row 0 the
    semantic token ids, rows 1.. the codebook indices; every value is exact in float32) and the float32 waveform
    [B, 1, NF*2048]: whole as `waveform.npy` when it has at most DUMP_WAV_SAMPLES samples, else a fixed seeded sample of
    them as `waveform_sample.npy` with their flat indices (float64) in `waveform_sample_index.npy`."""
    import numpy as np

    out_dir.mkdir(parents=True, exist_ok=True)
    np.save(out_dir / "codes.npy", codes.cpu().numpy().astype(np.float32))
    if wav is None:
        return
    flat = wav.float().flatten().cpu().numpy()
    if flat.size <= DUMP_WAV_SAMPLES:
        np.save(out_dir / "waveform.npy", flat.reshape(tuple(wav.shape)))
        return
    idx = np.sort(np.random.default_rng(0).choice(flat.size, DUMP_WAV_SAMPLES, replace=False))
    np.save(out_dir / "waveform_sample.npy", flat[idx])
    np.save(out_dir / "waveform_sample_index.npy", idx.astype(np.float64))


def _timed_events(fn, steps, warmup=1):
    for _ in range(warmup):
        out = fn()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(steps):
        out = fn()
    ev1.record()
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1) / steps, out


def voice_clone_bench(args):
    """BASELINE configs[4] (SURVEY §8(d) config 5), single GPU: every step encodes the 10 s reference clips,
    builds the prompts (text ids + the reference's VQ columns + text ids), generates 512 frames per utterance
    and decodes them to waveform -- all through the public API, host audio in, host waveform out. The stages are
    also timed one by one (device events, same inputs)."""
    from fish_speech_b200 import synthetic
    from fish_speech_b200.configs import S2PRO_IM_END_ID, s2pro_args
    from fish_speech_b200.models.dac.inference import load_codec_config
    from fish_speech_b200.models.dac.modded_dac import DAC
    from fish_speech_b200.models.text2semantic.inference import generate_batch
    from fish_speech_b200.models.text2semantic.llama import DualARTransformer

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    B, NF, REF_S = 8, 512, 10
    cfg = s2pro_args(max_seq_len=1024)
    w = synthetic.lm_state_dict(cfg, dev)
    w["embeddings.weight"][S2PRO_IM_END_ID] = 0
    model = DualARTransformer(cfg, w, device=dev, im_end_id=S2PRO_IM_END_ID)
    model.max_rows = 4096
    model.setup_caches(max_batch_size=B, max_seq_len=cfg.max_seq_len)
    del w
    eng = model.engine
    ccfg = load_codec_config("modded_dac_vq")
    dac = DAC(ccfg, synthetic.codec_state_dict(ccfg, dev), device=dev)
    g = torch.Generator().manual_seed(0)
    audio_host = (0.1 * torch.randn(B, 1, 44100 * REF_S, generator=g)).pin_memory()
    C = cfg.num_codebooks
    ta = torch.zeros(B, C + 1, 64, dtype=torch.int32)
    tb = torch.zeros(B, C + 1, 64, dtype=torch.int32)
    ta[:, 0] = torch.randint(0, 151643, (B, 64), generator=g, dtype=torch.int32)
    tb[:, 0] = torch.randint(0, 151643, (B, 64), generator=g, dtype=torch.int32)
    ta, tb = ta.to(dev), tb.to(dev)
    audio_lens = torch.full((B,), 44100 * REF_S, dtype=torch.long, device=dev)
    T_REF = -(-44100 * REF_S // 2048)  # every clip has the same length here: no per-utterance host sync

    def encode():
        return dac.encode(audio_host.to(dev, non_blocking=True), audio_lens)[0]  # [B, 10, 216]

    def prompts_of(codes):
        vq = torch.zeros(B, C + 1, T_REF, dtype=torch.int32, device=dev)
        vq[:, 0] = codes[:, 0, :T_REF].to(torch.int32) + cfg.semantic_begin_id
        vq[:, 1:] = codes[:, :, :T_REF].to(torch.int32)
        return list(torch.cat([ta, vq, tb], dim=2).unbind(0))

    def generate(prompts):
        return generate_batch(model=model, prompts=prompts, max_new_tokens=NF, temperature=0.7, top_p=0.7, top_k=1, seed=1)

    def step():
        prompts = prompts_of(encode())
        outs = generate(prompts)
        plen = prompts[0].shape[1]
        gen = torch.stack([o[1:, plen: plen + NF] for o in outs]).contiguous()
        return dac.from_indices(gen).cpu(), plen

    ms, (wav, plen) = _timed_events(step, args.steps, max(1, args.warmup))
    # ---- stage breakdown ----
    codes = encode()
    prompts = prompts_of(codes)
    sp = eng.sampling(0.7, 0.7, 1, 1)
    enc_ms, _ = _timed_events(encode, 3)

    def prefill():
        eng.reset()
        eng.prefill(prompts, list(range(B)), sp, do_sample=True)

    pre_ms, _ = _timed_events(prefill, 3)
    dec_ms, _ = _timed_events(lambda: eng.decode(B, 64, sp, use_graph=True), 2)
    dec_ms /= 64
    gen_codes = eng.buffer("out_tokens")[:B, 1:, :NF].contiguous()
    cod_ms, _ = _timed_events(lambda: dac.from_indices(gen_codes), 3)
    api_ms, _ = _timed_events(lambda: generate(prompts), 1)
    audio_s = B * NF * FRAME / SR
    v = audio_s / (ms / 1e3)
    kv_per_tok = cfg.n_layer * 2 * cfg.n_local_heads * cfg.head_dim * 2
    print(json.dumps({
        "metric": "audio-sec/s", "value": v, "unit": "audio-s/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": {"workload": f"voice-clone: batch-{B}, {REF_S} s reference audio -> encode -> {plen}-position prefill -> "
                               f"{NF} frames -> waveform, S2-Pro geometry", "frames_per_s": B * NF / (ms / 1e3),
                   "stages": ["codec_encode", "lm_prefill", "lm_decode", "codec_decode"],
                   "stage_ms": {"codec_encode_8x10s": enc_ms, "lm_prefill": pre_ms, "lm_decode_per_frame": dec_ms,
                                "lm_decode_511_frames": dec_ms * (NF - 1), "codec_decode": cod_ms,
                                "generate_batch_api_call": api_ms,
                                "sum_of_stages": enc_ms + pre_ms + dec_ms * (NF - 1) + cod_ms},
                   "decode_floor_ms_per_frame": (15.55e9 + B * (plen + NF / 2) * kv_per_tok) / (peaks()[0]["hbm_gbs"] * 1e9) * 1e3},
        "e2e": {"value": v, "unit": "audio-s/s", "h2d_bytes_per_step": audio_host.numel() * 4,
                "d2h_bytes_per_step": wav.numel() * 4},
    }))


def single_stream_bench(args):
    """BASELINE configs[1] (SURVEY §8(d) config 2): ONE 64-token prompt, greedy, 256 frames, LM stage: frames/s of a
    single stream against the weight-streaming floor (15.55 GB per frame whatever the batch)."""
    from fish_speech_b200 import synthetic
    from fish_speech_b200.configs import S2PRO_IM_END_ID
    from fish_speech_b200.models.text2semantic.inference import generate
    from fish_speech_b200.models.text2semantic.llama import DualARTransformer

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    cfg = s2pro_cfg()
    w = synthetic.lm_state_dict(cfg, dev)
    w["embeddings.weight"][S2PRO_IM_END_ID] = 0
    model = DualARTransformer(cfg, w, device=dev, im_end_id=S2PRO_IM_END_ID)
    model.setup_caches(max_batch_size=1, max_seq_len=cfg.max_seq_len)
    del w
    eng = model.engine
    prompt_host = make_prompts(cfg, 1, 42)[0].pin_memory()
    sp = eng.sampling(0.7, 0.7, 1, 42)
    NF = N_FRAMES

    def api():
        return generate(model=model, prompt=prompt_host.to(dev, non_blocking=True), max_new_tokens=NF, temperature=0.7,
                        top_p=0.7, top_k=1, seed=42).cpu()

    ms, out = _timed_events(api, args.steps, max(1, args.warmup))
    eng.reset()
    eng.prefill([prompt_host.to(dev)], [0], sp, do_sample=True)
    dec_ms, _ = _timed_events(lambda: eng.decode(1, 100, sp, use_graph=True), 2)
    dec_ms /= 100
    pk, _ = peaks()
    kv_per_tok = cfg.n_layer * 2 * cfg.n_local_heads * cfg.head_dim * 2
    floor_ms = (15.55e9 + (T_PROMPT + 120) * kv_per_tok) / (pk["hbm_gbs"] * 1e9) * 1e3
    v = NF * FRAME / SR / (ms / 1e3)
    print(json.dumps({
        "metric": "audio-sec/s", "value": v, "unit": "audio-s/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": {"workload": "S2-Pro 4B Dual-AR greedy decode, single 64-token prompt, 256 frames, LM stage, 1 GPU",
                   "frames_per_s": NF / (ms / 1e3), "codec_tokens_per_s": NF * cfg.num_codebooks / (ms / 1e3),
                   "ms_per_decode_frame": dec_ms, "hbm_floor_ms_per_frame": floor_ms, "hbm_frac": floor_ms / dec_ms,
                   "generated": list(out.shape)},
        "e2e": {"value": v, "unit": "audio-s/s", "h2d_bytes_per_step": prompt_host.numel() * 4,
                "d2h_bytes_per_step": out.numel() * 8},
    }))


def roundtrip_bench(args):
    """BASELINE configs[0] (SURVEY §8(d) config 1): Firefly VQ-GAN encode -> decode of 1 s of 44.1 kHz audio, host
    waveform in, host waveform out, beside the reference's CPU path (oracle/cpu_baseline.py codec) on the host cores."""
    from fish_speech_b200 import synthetic
    from fish_speech_b200.models.dac.inference import load_codec_config
    from fish_speech_b200.models.dac.modded_dac import DAC

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    ccfg = load_codec_config("modded_dac_vq")
    dac = DAC(ccfg, synthetic.codec_state_dict(ccfg, dev), device=dev)
    g = torch.Generator().manual_seed(0)
    wav_host = (0.1 * torch.randn(1, 1, 44100, generator=g)).pin_memory()

    def step():
        codes, lens = dac.encode(wav_host.to(dev, non_blocking=True))
        return dac.from_indices(codes).cpu(), codes

    ms, (wav, codes) = _timed_events(step, max(args.steps, 10), 3)
    enc_ms, _ = _timed_events(lambda: dac.encode(wav_host.to(dev)), 10, 2)
    dec_ms, _ = _timed_events(lambda: dac.from_indices(codes), 10, 2)
    cpu = None
    if not args.no_cpu_baseline:
        import time

        from oracle import codec_oracle as CO
        from oracle import cpu_baseline

        torch.set_num_threads(min(cpu_baseline.usable_cores(), 32))
        oc = CO.full_config()
        ow = CO.make_weights(oc, seed=6)
        with torch.inference_mode():
            CO.encode(ow, oc, wav_host.clone())  # warm-up
            t0 = time.perf_counter()
            c2, _ = CO.encode(ow, oc, wav_host.clone())
            t1 = time.perf_counter()
            CO.from_indices(ow, oc, c2)
            t2 = time.perf_counter()
        cpu = {"value": 1.0 / (t2 - t0), "unit": "audio-s/s", "cores": torch.get_num_threads(), "kind": "port",
               "sample": f"the same 1 s clip, fp32: encode {1e3 * (t1 - t0):.0f} ms + decode {1e3 * (t2 - t1):.0f} ms"}
    v = (codes.shape[-1] * FRAME / SR) / (ms / 1e3)
    print(json.dumps({
        "metric": "audio-sec/s", "value": v, "unit": "audio-s/s", "n_gpus": 1, "steps": max(args.steps, 10), "warmup": 3,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": {"workload": "Firefly VQ-GAN (391 M DAC) encode -> decode roundtrip, 1 s 44.1 kHz mono, batch 1",
                   "stage_ms": {"encode": enc_ms, "decode": dec_ms}, "codes": list(codes.shape)},
        "e2e": {"value": v, "unit": "audio-s/s", "h2d_bytes_per_step": wav_host.numel() * 4, "d2h_bytes_per_step": wav.numel() * 4},
        "cpu_baseline": cpu,
    }))


def stream_bench(args):
    """SURVEY §8(f).3: time to first audio of ONE utterance (64-token prompt, 256 frames) with the codec decoding every
    8 frames on a second CUDA stream while the LM keeps decoding (generate(frame_callback) + DAC.open_decode_stream),
    against decoding the codes after the LM has finished (the reference's order, inference_engine/__init__.py:84-119)."""
    import time

    from fish_speech_b200 import synthetic
    from fish_speech_b200.configs import S2PRO_IM_END_ID
    from fish_speech_b200.models.dac.inference import load_codec_config
    from fish_speech_b200.models.dac.modded_dac import DAC
    from fish_speech_b200.models.text2semantic.inference import generate
    from fish_speech_b200.models.text2semantic.llama import DualARTransformer

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    cfg = s2pro_cfg()
    w = synthetic.lm_state_dict(cfg, dev)
    w["embeddings.weight"][S2PRO_IM_END_ID] = 0
    model = DualARTransformer(cfg, w, device=dev, im_end_id=S2PRO_IM_END_ID)
    model.setup_caches(max_batch_size=1, max_seq_len=cfg.max_seq_len)
    del w
    ccfg = load_codec_config("modded_dac_vq")
    dac = DAC(ccfg, synthetic.codec_state_dict(ccfg, dev), device=dev)
    prompt = make_prompts(cfg, 1, 42)[0].to(dev)
    NF = N_FRAMES
    side = torch.cuda.Stream(device=dev)
    kw = dict(model=model, prompt=prompt, max_new_tokens=NF, temperature=0.7, top_p=0.7, top_k=1, seed=42)

    def streamed():
        st = dac.open_decode_stream(batch=1, max_frames=NF + 8)
        t0 = time.perf_counter()
        first, pieces = [None], []

        def cb(b, codes):
            with torch.cuda.stream(side):
                wav = st.push(codes[None].to(dev)).cpu()
            if first[0] is None:
                first[0] = time.perf_counter() - t0
            pieces.append(wav)

        y = generate(frame_callback=cb, **kw)
        total = time.perf_counter() - t0
        return first[0], total, torch.cat(pieces, dim=-1), y

    def after():
        t0 = time.perf_counter()
        y = generate(**kw)
        wav = dac.from_indices(y[None, 1:, T_PROMPT:-1].contiguous()).cpu()
        return time.perf_counter() - t0, wav

    for _ in range(2):
        streamed()
        after()
    fa, tot, wav_s, y = streamed()
    t_after, wav_a = after()
    same = wav_s.shape == wav_a.shape and float((wav_s - wav_a).abs().max()) < 1e-3
    print(json.dumps({
        "metric": "time-to-first-audio", "value": fa * 1e3, "unit": "ms", "n_gpus": 1, "steps": 1, "warmup": 2,
        "ms_per_step": tot * 1e3, "higher_is_better": False, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": {"workload": "1 utterance, 64-token prompt, 256 frames, codec decoded every 8 frames while the LM decodes",
                   "first_audio_ms_streaming": fa * 1e3, "total_ms_streaming": tot * 1e3,
                   "first_audio_ms_decode_after_lm": t_after * 1e3, "audio_s": (NF - 1) * FRAME / SR,
                   "same_waveform": bool(same)},
    }))


def serve_bench(args):
    """SURVEY 8(f).1: a queue of requests with RAGGED lengths (the fixed-length headline hides what the
    reference's one-request-at-a-time worker and a static batch both lose). 192 requests, 64-token prompts,
    64..256 frames each (seeded), greedy, LM stage only (the codec stage is the same work either way).
    Measured twice on the same requests: static batches of 32 in arrival order (`generate_batch`: a batch
    lasts as long as its longest request) and the slot scheduler (`ContinuousBatcher`, 32 slots)."""
    from fish_speech_b200 import synthetic
    from fish_speech_b200.configs import S2PRO_IM_END_ID, s2pro_args
    from fish_speech_b200.models.text2semantic.inference import generate_batch
    from fish_speech_b200.models.text2semantic.llama import DualARTransformer
    from fish_speech_b200.scheduler import ContinuousBatcher, SlotRequest

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    NREQ, SLOTS = 192, 32
    cfg = s2pro_args(max_seq_len=T_PROMPT + 256)
    w = synthetic.lm_state_dict(cfg, dev)
    w["embeddings.weight"][S2PRO_IM_END_ID] = 0  # lengths are set by the per-request budgets
    model = DualARTransformer(cfg, w, device=dev, im_end_id=S2PRO_IM_END_ID)
    model.max_rows = SLOTS * T_PROMPT
    model.setup_caches(max_batch_size=SLOTS, max_seq_len=cfg.max_seq_len)
    del w
    g = torch.Generator().manual_seed(7)
    lens = torch.randint(64, 257, (NREQ,), generator=g).tolist()
    prompts = [p.to(dev) for p in make_prompts(cfg, NREQ, 42)]
    audio_s = sum(lens) * FRAME / SR

    def static():
        outs = []
        for i in range(0, NREQ, SLOTS):
            n = max(lens[i:i + SLOTS])
            o = generate_batch(model=model, prompts=prompts[i:i + SLOTS], max_new_tokens=n, temperature=0.7,
                               top_p=0.7, top_k=1, seed=1)
            outs += [x[:, :T_PROMPT + k] for x, k in zip(o, lens[i:i + SLOTS])]
        return outs

    stats = {}

    def continuous():
        b = ContinuousBatcher(model, max_slots=SLOTS, frames_per_poll=8)
        reqs = [b.submit(SlotRequest(prompt=p, max_new_tokens=k, temperature=0.7, top_p=0.7, top_k=1, seed=1))
                for p, k in zip(prompts, lens)]
        b.run()
        stats["frames_run"], stats["occupancy"] = b.frames_run, b.slot_frames / max(1, b.frames_run * SLOTS)
        b.close()
        return [r.result for r in reqs]

    def timed(fn):
        for _ in range(max(1, min(args.warmup, 2))):
            out = fn()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(args.steps):
            out = fn()
        ev1.record()
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1) / args.steps, out

    ms_s, out_s = timed(static)
    ms_c, out_c = timed(continuous)
    same = all(torch.equal(a, b) for a, b in zip(out_s, out_c))
    v = audio_s / (ms_c / 1e3)
    print(json.dumps({
        "metric": "audio-sec/s", "value": v, "unit": "audio-s/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_c, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": {"workload": f"serve: {NREQ} queued requests, {T_PROMPT}-token prompts, 64..256 frames each "
                               f"(mean {sum(lens) / NREQ:.0f}), greedy, LM stage only, {SLOTS} slots, S2-Pro geometry",
                   "static_batches_audio_s_per_s": audio_s / (ms_s / 1e3), "static_ms": ms_s,
                   "continuous_over_static": ms_s / ms_c, "slot_occupancy": stats["occupancy"],
                   "decode_frames_run": stats["frames_run"], "identical_tokens": bool(same)},
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--frames", type=int, default=N_FRAMES)
    ap.add_argument("--batch", type=int, default=B_PER_GPU)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-codec", action="store_true", help="time the LM stages only")
    ap.add_argument("--profile-only", action="store_true", help="run the timed step once and exit (for ncu)")
    ap.add_argument("--workload", default="batch32", choices=["batch32", "voice-clone", "serve", "single", "roundtrip", "stream"],
                    help="batch32 = BASELINE configs[2] (the headline); voice-clone = configs[4]: 10 s reference "
                         "audio -> codec encode -> ~350-position prefill -> 512 frames -> waveform, batch 8")
    ap.add_argument("--dump-outputs", type=Path, metavar="DIR",
                    help="write the codes and waveform of the last timed step to DIR/<name>.npy (batch32, one GPU)")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and (args.workload != "batch32" or args.impl != "b200" or world > 1
                                          or args.profile_only):
        ap.error("--dump-outputs covers the batch32 workload of the b200 implementation on one GPU")
    workload = (f"batch-{args.batch} text->codec->wav, {T_PROMPT}-token prompts, {args.frames} codec frames/utt, "
                "S2-Pro 4B Dual-AR + 391M DAC codec geometry")

    if args.workload == "voice-clone" and args.impl != "reference":
        return voice_clone_bench(args)
    if args.workload == "serve" and args.impl != "reference":
        return serve_bench(args)
    if args.workload in ("single", "roundtrip", "stream") and args.impl != "reference":
        return {"single": single_stream_bench, "roundtrip": roundtrip_bench, "stream": stream_bench}[args.workload](args)
    if args.impl == "reference":
        if rank != 0:
            return
        r = cpu_reference(args.steps, args.warmup)
        cb = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}
        print(json.dumps({
            "impl": "reference", "metric": "audio-sec/s", "value": r["value"], "unit": "audio-s/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": workload, "stages": ["lm_prefill", "lm_decode", "codec_decode"],
                       "utterances": args.batch * world, "sampling": "greedy top_k=1 T=0.7 top_p=0.7",
                       "step": "bounded sample of the workload, see cpu_baseline.sample",
                       "measured": {k: r[k] for k in ("t_prefill_s", "t_frame_s", "t_codec_s", "frames_per_step",
                                                      "codec_frames_per_step")}},
            "cpu_baseline": cb,
            "e2e": {"value": r["value"], "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return

    import torch.distributed as dist

    from fish_speech_b200 import _lib
    from fish_speech_b200.models.text2semantic.inference import generate_batch
    from fish_speech_b200 import synthetic
    from fish_speech_b200.configs import S2PRO_IM_END_ID
    from fish_speech_b200.models.dac.inference import load_codec_config
    from fish_speech_b200.models.dac.modded_dac import DAC
    from fish_speech_b200.models.text2semantic.llama import DualARTransformer

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # stdout carries exactly ONE line, the JSON result: whatever NCCL prints while the communicator comes up (its
        # version banner at NCCL_DEBUG=VERSION / INFO goes to stdout) is sent to stderr; NCCL's settings are not touched
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    cfg = s2pro_cfg()
    B, NF = args.batch, args.frames
    # N > 1: rank 0 synthesises the checkpoint, the other ranks receive it over NCCL (NVLink) -- the start-up path of a
    # multi-GPU deployment (DESIGN.md section 6); outside the timed region
    weights = synthetic.lm_state_dict(cfg, dev) if rank == 0 else None
    weights_from = "synthesised on the device"
    if world > 1:
        from fish_speech_b200.parallel import broadcast_state_dict

        torch.cuda.synchronize()
        t0 = time.perf_counter()
        weights = broadcast_state_dict(weights, 0, dev)
        torch.cuda.synchronize()
        nbytes = sum(v.numel() * v.element_size() for v in weights.values())
        weights_from = f"rank 0 -> NCCL broadcast, {nbytes / 1e9:.2f} GB in {time.perf_counter() - t0:.2f} s"
    # fixed-length workload (SURVEY §8(d) config 2/3: "<|im_end|> bias set to -inf"): a zero head row gives
    # <|im_end|> the logit 0, which never beats the best of 4096 random semantic logits
    weights["embeddings.weight"][S2PRO_IM_END_ID] = 0
    model = DualARTransformer(cfg, weights, device=dev, im_end_id=S2PRO_IM_END_ID)
    model.max_rows = B * T_PROMPT
    model.setup_caches(max_batch_size=B, max_seq_len=cfg.max_seq_len)
    del weights
    eng = model.engine
    ccfg = load_codec_config("modded_dac_vq")
    with torch.cuda.device(dev):
        cw = synthetic.codec_state_dict(ccfg, dev)
        dac = DAC(ccfg, cw, device=dev)
        del cw
    stages = ["lm_prefill", "lm_decode"] + ([] if args.no_codec else ["codec_decode"])
    # utterance shard of this rank: utts[rank::world] of 32*world prompts (seeds 42..)
    prompts_host = [p.pin_memory() for p in make_prompts(cfg, B * world, 42)[rank::world]]
    prompts_dev = [p.to(dev) for p in prompts_host]
    sp = eng.sampling(0.7, 0.7, 1, 42)
    L = _lib.lib()

    def codec_stage():
        codes = eng.buffer("out_tokens")[:B, 1:, :NF].contiguous()
        return dac.from_indices(codes)

    last_wav = [None]  # waveform of the latest step_resident (--dump-outputs)

    def step_resident():
        eng.reset()
        eng.prefill(prompts_dev, list(range(B)), sp, do_sample=True)
        eng.decode(B, NF - 1, sp, use_graph=True)
        if not args.no_codec:
            last_wav[0] = codec_stage()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        for _ in range(steps):
            fn()
        ev1.record()
        barrier()
        ms = ev0.elapsed_time(ev1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    for _ in range(args.warmup):
        step_resident()
    if args.profile_only:
        step_resident()
        torch.cuda.synchronize()
        return
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    launches0 = _lib.launch_count()  # counts eager launches AND the kernels of every graph replay
    ms = timed(step_resident, args.steps)
    launches = _lib.launch_count() - launches0
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs is not None:  # before anything else reuses the engine's buffers
        dump_outputs(args.dump_outputs, eng.buffer("out_tokens")[:B, :, :NF], last_wav[0])
    ms_per_step = ms / args.steps
    audio_s = B * world * NF * FRAME / SR
    value = audio_s / (ms_per_step / 1e3)

    # ---- e2e through the public API: host prompts -> generate_batch -> codes on the host ----
    def step_e2e():
        outs = generate_batch(model=model, prompts=[p.to(dev, non_blocking=True) for p in prompts_host],
                              max_new_tokens=NF, temperature=0.7, top_p=0.7, top_k=1, seed=42)
        if args.no_codec:
            return [o[:, T_PROMPT:].cpu() for o in outs]
        # fixed-length workload (<|im_end|> cannot win with these weights): one padded codec batch
        codes = torch.stack([o[1:, T_PROMPT:T_PROMPT + NF] for o in outs]).contiguous()
        return dac.from_indices(codes).cpu()

    step_e2e()
    ms_e2e = timed(step_e2e, max(1, args.steps // 2)) / max(1, args.steps // 2)
    e2e_value = audio_s / (ms_e2e / 1e3)
    h2d = sum(p.numel() * p.element_size() for p in prompts_host) * world
    d2h = B * world * (cfg.num_codebooks + 1) * NF * 4 if args.no_codec else B * world * NF * FRAME * 4
    # ---- stage breakdown: prefill alone, decode frames alone (device-timed, same inputs) ----
    def prefill_only():
        eng.reset()
        eng.prefill(prompts_dev, list(range(B)), sp, do_sample=True)

    prefill_only()
    prefill_ms = timed(prefill_only, 3) / 3
    DEC_FRAMES = min(NF - 1, 128)
    decode_ms = timed(lambda: eng.decode(B, DEC_FRAMES, sp, use_graph=True), 1) / DEC_FRAMES  # per frame, context ~T+64
    codec = None
    if not args.no_codec:
        codec_stage()
        codec_ms = timed(codec_stage, 3) / 3
        flops = 2.0 * codec_decode_macs(ccfg, NF) * B
        codec = {"ms": codec_ms, "tflops": flops / (codec_ms / 1e3) / 1e12, "flop_per_step": flops}

    # ---- roofline of the dominant kernel (the weight-streaming step GEMM), measured live two ways:
    #  in-frame  = algorithmic bytes of one decode frame / device time of one decode frame of the timed run
    #              (everything between the GEMMs -- attention, sampling, dependency latency -- counts against it)
    #  replay    = the same 311 step GEMMs launched back to back without the kernels in between ----
    import ctypes as C

    wb, nl = C.c_double(), C.c_int()
    reps = 20
    _lib.check(L.fsb_lm_bench_gemms(eng.h, 2, C.byref(wb), C.byref(nl), torch.cuda.current_stream().cuda_stream))
    gemm_ms = timed(lambda: _lib.check(L.fsb_lm_bench_gemms(eng.h, reps, C.byref(wb), C.byref(nl),
                                                            torch.cuda.current_stream().cuda_stream)), 1)
    pk, pk_kind = peaks()
    gemm_gbs = wb.value * reps / (gemm_ms / 1e3) / 1e9
    # frame-level: algorithmic bytes per frame = weights + KV reads (B * L * 147456 B), SURVEY §8(d)
    kv_per_tok = cfg.n_layer * 2 * cfg.n_local_heads * cfg.head_dim * 2
    avg_L = T_PROMPT + NF / 2
    frame_bytes = wb.value + B * avg_L * kv_per_tok
    frame_ms = ms_per_step / NF  # includes the prefill and the codec, amortised
    dec_bytes = wb.value + B * (T_PROMPT + DEC_FRAMES / 2) * kv_per_tok
    dec_gbs = dec_bytes / (decode_ms / 1e3) / 1e9

    out = None
    if rank == 0:
        out = {
            "metric": "audio-sec/s", "value": value, "unit": "audio-s/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {
                "workload": workload, "stages": stages, "utterances": B * world,
                "frames_per_s": B * world * NF / (ms_per_step / 1e3),
                "codec_tokens_per_s": B * world * NF * cfg.num_codebooks / (ms_per_step / 1e3),
                "ms_per_frame": frame_ms, "ms_per_decode_frame": decode_ms, "prefill_ms": prefill_ms,
                "codec_ms": codec["ms"] if codec else None, "sampling": "greedy top_k=1 T=0.7 top_p=0.7",
                "l2_note": "inputs larger than L2: 9.1 GB of weights streamed per frame (126 MB L2)",
                "parallelism": f"replica x{world}, utts[rank::world]", "weights": weights_from,
                "step_hbm_frac": frame_bytes / (frame_ms / 1e3) / 1e9 / pk["hbm_gbs"],
            },
            "e2e": {"value": e2e_value, "unit": "audio-s/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e},
            "gpu_launches": int(launches),
            "roofline": {
                "bound": "hbm", "achieved": dec_gbs, "peak": pk["hbm_gbs"], "unit": "GB/s",
                "frac": dec_gbs / pk["hbm_gbs"], "traffic": ncu_traffic(), "peak_kind": pk_kind,
                "kernel": "step_gemm_kernel (tcgen05 + TMA weight streaming, host-scheduled stream-K, RMSNorm applied on "
                          "operand load; partials finished by the consuming kernels), in-frame: bytes of one decode frame "
                          "(weights + KV) / device time of one frame",
                "bytes_per_launch": dec_bytes / nl.value, "launches_per_frame": nl.value,
                "avg_launch_us": decode_ms * 1e3 / nl.value, "frame_bytes": dec_bytes, "frame_ms": decode_ms,
                "replay": {"achieved": gemm_gbs, "frac": gemm_gbs / pk["hbm_gbs"], "bytes_per_launch": wb.value / nl.value,
                           "launches": nl.value * reps, "avg_launch_us": gemm_ms * 1e3 / (nl.value * reps),
                           "note": "the same step GEMMs back to back, no attention / sampling kernels between them"},
            },
            "clocks": clk,
        }
        if codec is not None:
            pkv = pk.get("bf16_tflops_sustained", 1400.0)
            out["roofline_codec"] = {"bound": "tensor", "achieved": codec["tflops"], "peak": pkv, "unit": "TFLOP/s",
                                     "frac": codec["tflops"] / pkv, "traffic": None, "ms_per_step": codec["ms"],
                                     "kernel": "gemm_tc_kernel<BN,1> implicit-im2col conv GEMMs (tcgen05) + glue",
                                     "flop_per_step": codec["flop_per_step"]}
    if world > 1:
        dist.barrier()
    if rank == 0:
        if not args.no_cpu_baseline and world == 1:  # reported at N=1 only (rank 0's host cores)
            try:
                r = cpu_reference(3, 1)
                out["cpu_baseline"] = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}
            except Exception as e:  # pragma: no cover
                out["cpu_baseline"] = {"value": None, "error": repr(e)}
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
