"""The Qwen3 seam.  The reference's QwenAudioCausalKVEncoder and StreamingMelExtractor were driven with ragged chunk
schedules and every output recorded (oracle/make_golden_seams.py); the drop-ins, built the way callers build them from
the reference's objects (weights taken from its tower's state_dict, geometry read off its modules and attributes), must
reproduce every hidden state and mel frame and the state fields callers read.  The CPU oracle stands behind the engine
API."""
import os
import types

import numpy as np
import pytest
import torch

from oracle.make_golden_seams import MEL_APPENDS, QWEN_DROPIN, QWEN_ENCODER_ATTRS, QWEN_STATE_FIELDS

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _encoder_like_reference(dims, sd, g):
    """The reference encoder as the drop-in reads it: its tower module (the geometry tower its fixtures were recorded
    with) and the attributes it set from its config."""
    from oracle.make_golden_qwen import GeometryTower
    return types.SimpleNamespace(audio_tower=GeometryTower(dims, sd).eval(), config=types.SimpleNamespace(n_mels=int(g["n_mels"])),
                                 **{k: int(g[f"attr_{k}"]) for k in QWEN_ENCODER_ATTRS})


@pytest.mark.parametrize("name", QWEN_DROPIN)
def test_drop_in_encoder_equals_reference(name):
    from oracle.make_golden_qwen import mel_stream
    from oracle.qwen_oracle import QwenTowerOracle
    from whisperlivekit_b200.qwen_dims import QWEN_DIMS, synthetic_tower_state_dict
    from whisperlivekit_b200.qwen_plugin import B200QwenAudioCausalKVEncoder

    g = dict(np.load(os.path.join(GOLDEN, f"qwen_dropin_{name}.npz")))
    dims = QWEN_DIMS[name]
    schedule = [int(n) for n in g["schedule"]]
    ref = _encoder_like_reference(dims, synthetic_tower_state_dict(dims, seed=23), g)
    mine = B200QwenAudioCausalKVEncoder.from_reference(ref, engine_factory=lambda d, sd: QwenTowerOracle(d, sd))
    assert mine.dims == dims                                              # geometry recovered from the modules
    mels = torch.from_numpy(mel_stream(sum(schedule), dims.n_mels, seed=4))
    sm = mine.init_state()
    a = 0
    with torch.no_grad():
        for i, n in enumerate(schedule + [-1]):                           # -1: flush_pending()
            hm, sm = mine.flush_pending(sm) if n < 0 else mine.forward_chunk(mels[None, a: a + n], sm)
            a += max(n, 0)
            hr = g[f"hidden{i}"]
            assert tuple(hm.shape) == hr.shape
            if hr.size:
                assert float(np.abs(hm.numpy() - hr).max()) < 2e-5
            for f, want in zip(QWEN_STATE_FIELDS, g[f"state{i}"]):
                if n >= 0 or f == "emitted_steps":
                    assert getattr(sm, f) == int(want), f
        assert sm.pending_frames == 0
    assert mine.right_context_frames == int(g["right_context_frames"])
    assert mine.output_steps_for_mel_frames(195) == int(g["output_steps_195"])


def test_drop_in_mel_extractor_equals_reference():
    """StreamingMelExtractor (reference, over the real Hugging Face featurizer) vs the drop-in over the engine API
    (CPU oracle behind it): same frames per append / flush, same values."""
    from oracle.make_golden_qwen_mel import speechlike
    from oracle.qwen_oracle import QwenTowerOracle
    from whisperlivekit_b200.qwen_dims import QWEN_DIMS, synthetic_tower_state_dict
    from whisperlivekit_b200.qwen_plugin import B200StreamingMelExtractor

    g = dict(np.load(os.path.join(GOLDEN, "qwen_mel_dropin.npz")))
    dims = QWEN_DIMS["qnano"]
    eng = QwenTowerOracle(dims, synthetic_tower_state_dict(dims, seed=1))
    eng.load_mel_filters()
    mine = B200StreamingMelExtractor(eng, eng.open_session())
    audio = speechlike(16000 * 4, seed=77)
    a = 0
    for i, n in enumerate(MEL_APPENDS + (-1,)):                           # -1: flush()
        m = mine.flush() if n < 0 else mine.append(audio[a: a + n])
        a += max(n, 0)
        assert (m is None) == bool(g[f"none{i}"])
        if m is not None:
            r = g[f"mel{i}"]
            assert tuple(m.shape) == r.shape and float(np.abs(m.numpy() - r).max()) < 5e-5
        assert mine.emitted_frames == int(g[f"emitted{i}"])
    assert mine.emitted_frames == a // 160
