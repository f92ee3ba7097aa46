#!/usr/bin/env python
"""Build container only: fixtures recorded from the REFERENCE for the tests of the drop-in seams, so that those tests
compare against the reference without importing it.

    python oracle/make_golden_seams.py <WhisperLiveKit checkout>
        # -> tests/golden/{alignment_heads,diar_reference,qwen_mel_dropin,qwen_dropin_<name>}.npz

  alignment_heads  the reference's _ALIGNMENT_HEADS table (whisper/__init__.py), decoded to boolean masks per model.
  diar_reference   SortformerDiarizationOnline._process_predictions on the 40 seeded random cases of
                   tests/test_diarization.py (NeMo stubbed out, as the reference's own tests do).
  qwen_mel_dropin  StreamingMelExtractor over the Hugging Face featurizer on the append schedule of
                   tests/test_qwen_plugin_reference.py: every frame of every append.
  qwen_dropin_*    QwenAudioCausalKVEncoder (the tower of make_golden_qwen.py, seed 23) on the same schedule: every hidden
                   state, the state fields callers read, and the encoder attributes the drop-in reads its geometry
                   from.
"""
import ast
import base64
import gzip
import importlib
import importlib.machinery
import os
import re
import sys
import threading
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
REF = os.path.abspath(sys.argv[1]) if __name__ == "__main__" else None
GOLDEN = os.path.join(ROOT, "tests", "golden")

# the random diarization cases and the Qwen append schedules the tests replay (they import these)
DIAR_TRIALS = 40
MEL_APPENDS = (100, 150, 4000, 333, 4000, 0, 12000, 4001)
QWEN_DROPIN = ("qnano", "qnano-chunk", "qnano-tail", "qnano-tail-bidir")
QWEN_STATE_FIELDS = ("frames_seen", "emitted_steps", "pending_frames", "last_input_frames", "last_recomputed_frames",
                     "last_recomputed_context_frames", "mutable_steps")
QWEN_ENCODER_ATTRS = ("chunk_frames", "block_frames", "left_context_steps", "block_bidirectional", "mutable_tail_steps")


def diar_cases():
    """The seeded random post-processing cases: (predictions, max_speakers, len_prediction, chunk_index, time offset)."""
    rng = np.random.default_rng(5)
    for trial in range(DIAR_TRIALS):
        n_spk = 4
        T = int(rng.integers(1, 60))
        preds = rng.random((T, n_spk)).astype(np.float32)
        if trial % 3 == 0:                                              # long runs + exact ties
            preds = np.repeat(np.round(preds[: max(1, T // 4)], 1), 4, axis=0)[:T]
        cap = int(rng.integers(1, 5))
        lp = None if trial % 2 == 0 else int(rng.integers(1, T + 1))
        chunk, gto = int(rng.integers(0, 50)), float(rng.choice([0.0, 1.37, 12.5]))
        yield preds, cap, lp, chunk, gto


def _stub_soundfile():
    if "soundfile" not in sys.modules:
        m = types.ModuleType("soundfile")
        m.__spec__ = importlib.machinery.ModuleSpec("soundfile", loader=None)
        sys.modules["soundfile"] = m


def alignment_heads():
    from whisperlivekit_b200.dims import ALIGNMENT_HEADS, DIMS
    src = open(os.path.join(REF, "whisperlivekit", "whisper", "__init__.py")).read()
    dumps = ast.literal_eval(re.search(r"_ALIGNMENT_HEADS = (\{.*?\n\})", src, re.S).group(1))
    out = {}
    for k in ALIGNMENT_HEADS:
        d = DIMS[k]
        out[k] = np.frombuffer(gzip.decompress(base64.b85decode(dumps[k])), dtype=bool).reshape(d.n_text_layer, d.n_text_head)
    return out


def diar_reference():
    sys.path.insert(0, REF)
    _stub_soundfile()
    for name in ("nemo", "nemo.collections", "nemo.collections.asr", "nemo.collections.asr.models", "nemo.collections.asr.modules"):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["nemo.collections.asr.models"].SortformerEncLabelModel = object
    sys.modules["nemo.collections.asr.modules"].AudioToMelSpectrogramPreprocessor = object
    sb = importlib.import_module("whisperlivekit.diarization.sortformer_backend")
    segs, offsets, lps = [], [0], []
    for preds, cap, lp, chunk, gto in diar_cases():
        online = object.__new__(sb.SortformerDiarizationOnline)
        online.total_preds = torch.tensor(preds[None], dtype=torch.float32)
        online.max_speakers = cap
        online._len_prediction = lp
        online.chunk_duration_seconds = 0.96
        online.segment_lock = threading.Lock()
        online._chunk_index = chunk
        online.global_time_offset = gto
        got = [(int(s.speaker), s.start, s.end) for s in online._process_predictions()]
        segs += got
        offsets.append(len(segs))
        lps.append(online._len_prediction)
    seg = np.asarray(segs, np.float64).reshape(-1, 3)
    return dict(speaker=seg[:, 0].astype(np.int64), start=seg[:, 1], end=seg[:, 2], offsets=np.asarray(offsets, np.int64),
                len_prediction=np.asarray(lps, np.int64))


def qwen_mel_dropin():
    sys.path.insert(0, os.path.join(REF, "third_party", "qwen3-asr-causal", "src"))
    from transformers import WhisperFeatureExtractor
    from qwen3_asr_causal.features import StreamingMelExtractor
    from oracle.make_golden_qwen_mel import speechlike
    ref = StreamingMelExtractor(WhisperFeatureExtractor(feature_size=128))
    audio = speechlike(16000 * 4, seed=77)
    rec, a = {}, 0
    for i, n in enumerate(MEL_APPENDS + (-1,)):                         # -1: flush()
        r = ref.flush() if n < 0 else ref.append(audio[a: a + n])
        a += max(n, 0)
        rec[f"none{i}"] = np.asarray(r is None)
        if r is not None:
            rec[f"mel{i}"] = r.numpy().astype(np.float32)
        rec[f"emitted{i}"] = np.asarray(ref.emitted_frames, np.int64)
    return rec


def qwen_dropin(name):
    sys.path.insert(0, os.path.join(REF, "third_party", "qwen3-asr-causal", "src"))
    from oracle.make_golden_qwen import SCHEDULE, TAIL_SCHEDULE, mel_stream, reference_encoder
    from whisperlivekit_b200.qwen_dims import QWEN_DIMS, synthetic_tower_state_dict
    dims = QWEN_DIMS[name]
    schedule = TAIL_SCHEDULE if dims.mutable_tail_steps else SCHEDULE
    ref = reference_encoder(dims, synthetic_tower_state_dict(dims, seed=23))
    mels = torch.from_numpy(mel_stream(sum(schedule), dims.n_mels, seed=4))
    rec = dict(schedule=np.asarray(schedule, np.int64), n_mels=np.asarray(int(ref.config.n_mels), np.int64),
               right_context_frames=np.asarray(ref.right_context_frames, np.int64),
               output_steps_195=np.asarray(ref.output_steps_for_mel_frames(195), np.int64),
               **{f"attr_{k}": np.asarray(int(getattr(ref, k)), np.int64) for k in QWEN_ENCODER_ATTRS})
    s, a = ref.init_state(), 0
    with torch.no_grad():
        for i, n in enumerate(schedule + [-1]):                           # -1: flush_pending()
            h, s = ref.flush_pending(s) if n < 0 else ref.forward_chunk(mels[None, a: a + n], s)
            a += max(n, 0)
            rec[f"hidden{i}"] = h.numpy().astype(np.float32)
            rec[f"state{i}"] = np.asarray([int(getattr(s, f)) for f in QWEN_STATE_FIELDS], np.int64)
    return rec


def main():
    _stub_soundfile()
    records = dict(alignment_heads=alignment_heads(), diar_reference=diar_reference(),
                   qwen_mel_dropin=qwen_mel_dropin(), **{f"qwen_dropin_{n}": qwen_dropin(n) for n in QWEN_DROPIN})
    for name, rec in records.items():
        path = os.path.join(GOLDEN, f"{name}.npz")
        np.savez_compressed(path, **rec)
        print(name, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
