"""Needs the reference package staged under oracle/_ref by build(): the LocalAgreement seam.  The reference's
unchanged whisper.transcribe() (DecodingTask, temperature fallback, timestamp rules, find_alignment + DTW) runs over
B200TranscribeModel; with the CPU oracle behind the engine API the result must equal what the same
transcribe() produces over the reference's own torch Whisper on the same weights and audio."""
import numpy as np
import pytest
import torch

from golden_util import case_setup

pytestmark = pytest.mark.reference


def _import_reference():
    from oracle import stage_reference
    stage_reference.import_staged_reference()


def _ref_model(dims, sd, heads):
    from oracle.make_golden import build_reference_model
    return build_reference_model(dims, sd, heads)


@pytest.mark.parametrize("name", ["micro", "microml"])
def test_transcribe_over_b200_model_equals_reference(name):
    _import_reference()
    from oracle import whisper_oracle as wo
    from whisperlivekit.whisper.transcribe import transcribe
    from whisperlivekit_b200.localagreement import B200WhisperASR

    g, dims, sd, audio, heads = case_setup(name)
    kw = dict(language="en", initial_prompt="", condition_on_previous_text=True, word_timestamps=True,
              temperature=(0.0,), no_speech_threshold=None, logprob_threshold=None, compression_ratio_threshold=None)
    torch.manual_seed(0)
    ref = transcribe(_ref_model(dims, sd, heads), audio, **kw)
    asr = B200WhisperASR(wo.OracleEngine(dims, sd, heads), lan="en")
    asr.transcribe_kargs = {k: v for k, v in kw.items() if k in ("temperature", "no_speech_threshold",
                                                                 "logprob_threshold", "compression_ratio_threshold")}
    torch.manual_seed(0)
    got = asr.transcribe(audio, init_prompt="")
    assert [s["tokens"] for s in got["segments"]] == [s["tokens"] for s in ref["segments"]]
    assert got["text"] == ref["text"]
    rw = [(w["word"], round(w["start"], 2), round(w["end"], 2)) for s in ref["segments"] for w in s["words"]]
    gw = [(w["word"], round(w["start"], 2), round(w["end"], 2)) for s in got["segments"] for w in s["words"]]
    assert gw == rw
    rp = [w["probability"] for s in ref["segments"] for w in s["words"]]
    gp = [w["probability"] for s in got["segments"] for w in s["words"]]
    np.testing.assert_allclose(gp, rp, rtol=1e-4, atol=1e-6)
    assert len(asr.ts_words(got)) == len(rw)
    assert asr.segments_end_ts(got) == [s["end"] for s in ref["segments"]]
    # the word-timestamp pass reused the segment's encoder output instead of encoding the same mel twice,
    # and median filter / DTW went through the engine's entry points (install_native_timing)
    assert asr.model.encoder_reuses == asr.model.encoder_calls >= 1
    import whisperlivekit.whisper.timing as timing
    assert hasattr(timing, "_b200_saved")
    from whisperlivekit_b200.localagreement import uninstall_native_timing
    uninstall_native_timing()


def test_transcribe_with_beam_search_equals_reference():
    """whisper.transcribe(beam_size=3): DecodingTask's beam rows (decoding.py:728) become forked sessions and
    PyTorchInference.rearrange_kv_cache (decoding.py:165-170) lands in gather_decoder; segments, tokens and word
    timings must equal the reference's over its own torch Whisper."""
    _import_reference()
    from oracle import whisper_oracle as wo
    from whisperlivekit.whisper.transcribe import transcribe
    from whisperlivekit_b200.localagreement import B200WhisperASR, uninstall_native_timing

    g, dims, sd, audio, heads = case_setup("micro")
    kw = dict(language="en", initial_prompt="", condition_on_previous_text=True, word_timestamps=True,
              temperature=(0.0,), beam_size=3, no_speech_threshold=None, logprob_threshold=None,
              compression_ratio_threshold=None)
    ref = transcribe(_ref_model(dims, sd, heads), audio, **kw)
    asr = B200WhisperASR(wo.OracleEngine(dims, sd, heads), lan="en")
    asr.transcribe_kargs = {k: v for k, v in kw.items() if k in ("temperature", "beam_size", "no_speech_threshold",
                                                                 "logprob_threshold", "compression_ratio_threshold")}
    got = asr.transcribe(audio, init_prompt="")
    uninstall_native_timing()
    assert [s["tokens"] for s in got["segments"]] == [s["tokens"] for s in ref["segments"]]
    rw = [(w["word"], round(w["start"], 2), round(w["end"], 2)) for s in ref["segments"] for w in s["words"]]
    gw = [(w["word"], round(w["start"], 2), round(w["end"], 2)) for s in got["segments"] for w in s["words"]]
    assert gw == rw
    assert len(asr.model._forks) == 2 and asr.model.gathers > 0
