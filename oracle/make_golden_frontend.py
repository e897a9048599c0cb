"""Record the reference's CPU prompt builder as driven by the generate_long plan (test infrastructure; needs the
reference checkout):

    python -m oracle.make_golden_frontend

Runs the plan of tests/test_engine_cpu.py (drive_generate_long_plan) with the UNMODIFIED fish_speech.conversation /
content_sequence and stores, for every prompt the plan asks for, the conversation it handed the builder (as the plan
constructed it) and the builder's encoded prompt in tests/golden/generate_long_frontend.npz. The CPU suite replays
that run without the reference."""
from __future__ import annotations

import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from oracle import ref_stubs as R  # noqa: E402

GOLD = ROOT / "tests" / "golden" / "generate_long_frontend.npz"


def main():
    if R.REF_ROOT not in sys.path:
        sys.path.insert(0, R.REF_ROOT)
    from fish_speech.content_sequence import TextPart, VQPart
    from fish_speech.conversation import Conversation, Message

    import fish_speech_b200.models.text2semantic.inference as inf
    from tests import test_engine_cpu as T

    calls = []

    def tagged(cls, kind):
        def make(**kw):
            obj = cls(**kw)
            obj.frontend_call = (kind, kw)
            return obj

        return make

    class RecordingConversation(Conversation):
        def encode_for_inference(self, tokenizer, num_codebooks, **kw):
            out = super().encode_for_inference(tokenizer, num_codebooks=num_codebooks, **kw)
            assert out[1] is None and out[2] is None, "no audio parts in this conversation"
            calls.append((T.frontend_conversation_json(self.messages), out[0].numpy().copy()))
            return out

    inf._reference_frontend = lambda: (tagged(TextPart, "TextPart"), tagged(VQPart, "VQPart"), RecordingConversation,
                                       tagged(Message, "Message"))
    tok = T._ByteTokenizer()
    prompts, _, _ = T.drive_generate_long_plan(tok)
    assert len(prompts) == len(calls) >= 2
    out = {"conversations": np.array([c for c, _ in calls]), "num_codebooks": np.int64(10),
           "tokenizer_special": np.array(json.dumps(tok.special))}
    for k, (_, enc) in enumerate(calls):
        out[f"encoded_{k}"] = enc
    GOLD.parent.mkdir(parents=True, exist_ok=True)
    np.savez_compressed(GOLD, **out)
    print(f"{GOLD}: {len(calls)} prompts, lengths {[e.shape[1] for _, e in calls]}")


if __name__ == "__main__":
    main()
