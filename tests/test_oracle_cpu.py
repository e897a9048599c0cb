"""CPU suite: the oracle against the committed outputs of the REAL reference (tests/golden/*.npz, written
by oracle/make_golden.py), host logic, and the C-ABI symbol table.  No GPU compute."""
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import lm_oracle as O
from tests.lm_util import load_golden

GOLD = Path(__file__).parent / "golden"
LM_CASES = sorted(p.name for p in GOLD.glob("lm_*.npz"))


def test_golden_fixtures_present():
    assert len(LM_CASES) >= 4


@pytest.mark.parametrize("name", LM_CASES)
def test_lm_oracle_matches_reference_golden(name):
    cfg, w, z = load_golden(GOLD / name)
    st = O.setup(cfg, w)
    prompt = torch.from_numpy(z["prompt"])
    traces = []
    torch.manual_seed(int(z["rng_seed"]))
    got = O.generate(st, prompt, int(z["new_frames"]), temperature=float(z["temperature"]),
                     top_p=float(z["top_p"]), top_k=int(z["top_k"]), traces=traces)
    assert np.array_equal(got.numpy(), z["ref_tokens"]), "oracle tokens differ from the reference's"
    logits = torch.stack([t["slow_logits"] for t in traces]).numpy().astype(np.float32)
    assert np.array_equal(logits, z["ref_slow_logits"])


def test_oracle_prompt_too_long_raises():
    cfg = O.tiny_config()
    w = O.make_weights(cfg, seed=1)
    st = O.setup(cfg, w)
    with pytest.raises(ValueError):
        O.generate(st, torch.zeros(cfg.num_codebooks + 1, cfg.max_seq_len, dtype=torch.long), 4)


def test_logits_to_probs_keeps_rank0_and_respects_topk():
    logits = torch.tensor([0.1, 3.0, 2.0, -1.0, 2.5]).bfloat16()
    p = O.logits_to_probs(logits, torch.tensor(1.0).bfloat16(), torch.tensor(0.01).bfloat16(), 3)
    assert p.argmax().item() == 1 and (p > 0).sum().item() == 1  # tiny top_p: only rank 0 survives
    p = O.logits_to_probs(logits, torch.tensor(1.0).bfloat16(), torch.tensor(1.0).bfloat16(), 2)
    assert set(torch.nonzero(p > 0).flatten().tolist()) == {1, 4}


def test_abi_exports_every_declared_symbol():
    from fish_speech_b200 import _lib

    L = _lib.lib()
    names = _lib.exported_symbols()
    assert len(names) >= 10
    missing = [n for n in names if not hasattr(L, n)]
    assert not missing, f"libfishb200.so lacks {missing}"


_WITHOUT_GPU = """
import os
import sys

sys.path.insert(0, os.getcwd())
import pytest
import torch
from fish_speech_b200 import _lib
from fish_speech_b200.models.text2semantic.llama import DualARTransformer
from oracle import lm_oracle as O
from tests.lm_util import model_args

assert not torch.cuda.is_available()
cfg = O.tiny_config()
m = DualARTransformer(model_args(cfg), O.make_weights(cfg, seed=1), im_end_id=cfg.im_end_id)
with pytest.raises(_lib.FsbError):
    m.setup_caches(1, cfg.max_seq_len)
print("failed loudly")
"""


def test_product_fails_loudly_without_gpu():
    """Run in a child process that sees no CUDA device, so that machines with a GPU check it too."""
    import os
    import subprocess
    import sys

    root = Path(__file__).resolve().parent.parent
    r = subprocess.run([sys.executable, "-c", _WITHOUT_GPU], cwd=root, env={**os.environ, "CUDA_VISIBLE_DEVICES": ""},
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "failed loudly" in r.stdout, r.stdout + r.stderr


def test_config_parsing_fish_qwen3_omni(tmp_path):
    import json

    from fish_speech_b200.models.text2semantic.llama import BaseModelArgs, DualARModelArgs

    cfgd = {
        "model_type": "fish_qwen3_omni", "semantic_start_token_id": 151678, "semantic_end_token_id": 155773,
        "text_config": {"vocab_size": 155776, "n_layer": 36, "n_head": 32, "n_local_heads": 8, "head_dim": 128,
                        "dim": 2560, "intermediate_size": 9728, "rope_base": 1000000, "norm_eps": 1e-6,
                        "max_seq_len": 32768, "attention_qk_norm": True, "tie_word_embeddings": True},
        "audio_decoder_config": {"vocab_size": 4096, "num_codebooks": 10, "n_layer": 4, "dim": 2560, "n_head": 32,
                                 "n_local_heads": 8, "head_dim": 128, "intermediate_size": 9728},
    }
    (tmp_path / "config.json").write_text(json.dumps(cfgd))
    a = BaseModelArgs.from_pretrained(str(tmp_path))
    assert isinstance(a, DualARModelArgs)
    assert a.scale_codebook_embeddings and a.norm_fastlayer_input
    assert (a.dim, a.n_layer, a.n_local_heads, a.codebook_size, a.num_codebooks, a.n_fast_layer) == (2560, 36, 8, 4096, 10, 4)
    assert a.fast_attention_qk_norm is True  # inherits attention_qk_norm when the decoder config is silent


def test_key_remap_and_qkv_fusion():
    from fish_speech_b200.models.text2semantic.llama import _fuse_qkv, _remap_fish_qwen3_omni_keys

    w = {"text_model.model.layers.0.attention.wq.weight": torch.ones(4, 2),
         "text_model.model.layers.0.attention.wk.weight": torch.ones(2, 2) * 2,
         "text_model.model.layers.0.attention.wv.weight": torch.ones(2, 2) * 3,
         "audio_decoder.codebook_embeddings.weight": torch.zeros(1),
         "audio_decoder.layers.0.ffn_norm.weight": torch.zeros(1)}
    r = _fuse_qkv(_remap_fish_qwen3_omni_keys(w))
    assert r["layers.0.attention.wqkv.weight"].shape == (8, 2)
    assert "codebook_embeddings.weight" in r and "fast_layers.0.ffn_norm.weight" in r


def test_text_batching_helpers():
    from fish_speech_b200.models.text2semantic.inference import group_turns_into_batches, split_text_by_speaker

    turns = split_text_by_speaker("<|speaker:0|>hello<|speaker:1|>hi there<|speaker:0|>bye")
    assert turns == ["<|speaker:0|>hello", "<|speaker:1|>hi there", "<|speaker:0|>bye"]
    assert group_turns_into_batches(turns, max_speakers=2, max_bytes=1000) == ["\n".join(turns[:2]), turns[2]]
    assert len(group_turns_into_batches(turns, max_speakers=5, max_bytes=20)) == 3


@pytest.mark.parametrize("tag", ["first", "mid"])
def test_oracle_stop_semantics_match_reference_golden(tag):
    """generate()'s <|im_end|> handling against outputs of the REAL reference (oracle/make_golden_stop.py):
    'first' = <|im_end|> as the prefill's token is not tested, the loop stops on the next one (inference.py:336-352,
    :233); 'mid' = a sampled run (same torch RNG stream) that draws <|im_end|> a few frames in and stops there."""
    from oracle import lm_oracle as O
    from tests.lm_util import make_prompt

    z = np.load(GOLD / "ref_stop_cases.npz")
    cfg = O.tiny_config()
    w = O.make_weights(cfg, seed=int(z["weight_seed"]), head_gain=float(z["head_gain"]))
    w["embeddings.weight"][cfg.im_end_id] = (w["embeddings.weight"][int(z[f"{tag}_src_token"])].float()
                                             * float(z[f"{tag}_gain"])).bfloat16()
    prompt = torch.from_numpy(z["prompt"])
    assert torch.equal(prompt, make_prompt(cfg, int(z["weight_seed"]), prompt.shape[1]))
    ref = torch.from_numpy(z[f"{tag}_ref_tokens"])
    torch.manual_seed(int(z[f"{tag}_rng_seed"]))
    got = O.generate(O.setup(cfg, w), prompt, int(z["max_new_tokens"]), temperature=float(z[f"{tag}_temperature"]),
                     top_p=float(z[f"{tag}_top_p"]), top_k=int(z[f"{tag}_top_k"]))
    assert torch.equal(got.to(torch.int32), ref)
    T = prompt.shape[1]
    hits = (ref[0, T:] == cfg.im_end_id).nonzero().flatten().tolist()
    assert ref.shape[1] < T + int(z["max_new_tokens"]) and ref[0, -1].item() == cfg.im_end_id
    assert hits == ([0, 1] if tag == "first" else [ref.shape[1] - T - 1])


# codec_tiny.npz was recorded with 8 intra-op CPU threads. The fp32 convolutions split their sums by thread count, so
# another count rounds the waveform differently in the last bits: the oracle is run with the recording's count.
GOLDEN_CODEC_THREADS = 8


def test_codec_oracle_matches_reference_golden_tiny():
    """oracle/codec_oracle.py against the committed outputs of the REAL reference codec (oracle/make_golden_codec.py):
    fp32 decode waveform bit-identical, encode codes identical (tiny geometry: runs in seconds)."""
    from oracle import codec_oracle as CO

    z = np.load(GOLD / "codec_tiny.npz")
    cfg = CO.tiny_config()
    w = CO.make_weights(cfg, seed=int(z["weight_seed"]))
    threads = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_CODEC_THREADS)
    try:
        with torch.inference_mode():
            wav = CO.from_indices(w, cfg, torch.from_numpy(z["codes"]).long())
            codes, lens = CO.encode(w, cfg, torch.from_numpy(z["audio"]), torch.from_numpy(z["lens"]))
    finally:
        torch.set_num_threads(threads)
    assert np.array_equal(wav.numpy(), z["ref_wav"]), "oracle waveform differs from the reference's"
    assert np.array_equal(codes.numpy().astype(np.int32), z["ref_codes"])
    assert np.array_equal(lens.numpy(), z["ref_lens"])


def test_codec_oracle_matches_reference_golden_full_encode():
    """Full 391 M-parameter geometry, BASELINE config #1 input (1 s of audio): the oracle's codes equal the real
    reference's (the decode at this size is checked on the GPU box against `ref_wav`)."""
    from oracle import codec_oracle as CO

    f = GOLD / "codec_full_1s.npz"
    if not f.exists():
        pytest.skip("full-size fixture not committed")
    z = np.load(f)
    cfg = CO.full_config()
    w = CO.make_weights(cfg, seed=int(z["weight_seed"]))
    with torch.inference_mode():
        codes, lens = CO.encode(w, cfg, torch.from_numpy(z["audio"]), torch.from_numpy(z["lens"]))
    assert np.array_equal(codes.numpy().astype(np.int32), z["ref_codes"])
    assert np.array_equal(lens.numpy(), z["ref_lens"])


def test_w13_interleave_layout():
    """Host side of the SwiGLU-in-epilogue weight layout (include/fishb200.h d_w13): row (f>>6)*128 + ((f>>4)&3)*32 +
    (f&15) holds w1[f], 16 rows further w3[f]; the hidden size is padded to a multiple of 64 with zero rows."""
    from fish_speech_b200.engine import interleave_w13

    I, D = 80, 8
    w1 = torch.arange(I * D, dtype=torch.float32).view(I, D)
    w3 = -w1 - 1
    m = interleave_w13(w1, w3)
    assert m.shape == (256, D)
    for f in (0, 15, 16, 63, 64, 79):
        r = (f >> 6) * 128 + ((f >> 4) & 3) * 32 + (f & 15)
        assert torch.equal(m[r], w1[f]) and torch.equal(m[r + 16], w3[f])
    used = {(f >> 6) * 128 + ((f >> 4) & 3) * 32 + (f & 15) + o for f in range(I) for o in (0, 16)}
    assert all(float(m[r].abs().sum()) == 0 for r in range(256) if r not in used)
