"""CPU: the Silero VAD oracle against probabilities recorded from the reference's scripted model
(oracle/make_golden_vad.py): seeded weights everywhere; with the trained weights where build() staged the reference
package under oracle/_ref."""
import os

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


def _audio():
    from whisperlivekit_b200.weights import synthetic_audio
    return np.concatenate([synthetic_audio(2.0, seed=31), np.zeros(8000, np.float32), 0.3 * synthetic_audio(1.5, seed=32)])


def test_vad_oracle_matches_reference_model_with_seeded_weights():
    from oracle.vad_oracle import VadOracle, synthetic_vad_state_dict
    g = dict(np.load(os.path.join(HERE, "golden", "vad.npz")))
    audio, n = _audio(), int(g["n_windows"])
    o = VadOracle(synthetic_vad_state_dict(seed=9))
    s = o.open_session()
    probs = np.concatenate([o.forward([s], [audio[i * 512:(i + 1) * 512]]) for i in range(n)])
    assert np.abs(probs - g["probs_seeded"]).max() < 2e-5
    assert probs.min() < 0.3 and probs.max() > 0.7                      # the fixture exercises both sides of a threshold


@pytest.mark.reference
def test_vad_oracle_matches_reference_model_with_trained_weights():
    import torch
    from oracle.stage_reference import TARGET
    from oracle.vad_oracle import VadOracle
    g = dict(np.load(os.path.join(HERE, "golden", "vad.npz")))
    m = torch.jit.load(os.path.join(TARGET, "whisperlivekit", "silero_vad_models", "silero_vad.jit"), map_location="cpu")
    o = VadOracle({k: v.numpy() for k, v in m.state_dict().items()})
    audio, n = _audio(), int(g["n_windows"])
    a, b = o.open_session(), o.open_session()
    probs = np.stack([o.forward([a, b], [audio[i * 512:(i + 1) * 512]] * 2) for i in range(n)])
    assert np.abs(probs[:, 0] - g["probs_trained"]).max() < 2e-5 and np.array_equal(probs[:, 0], probs[:, 1])
