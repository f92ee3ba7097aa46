"""Diarization post-processing (SURVEY.md 8f-4, reference sortformer_backend.py:313-363).
CPU: oracle/diar_oracle.py against the known answers of the reference's own tests (the reference project's
tests/test_sortformer_max_speakers.py:78-125, 183-215) and against the reference's method itself on random predictions
(recorded in tests/golden/diar_reference.npz).  GPU: the device run-length kernel (wlk_diar_segments, through the
C ABI) against the oracle, bit-exact (integer work)."""
import os

import numpy as np
import pytest

from oracle import diar_oracle as do

P1 = [[0.90, 0.10, 0.20, 0.05], [0.10, 0.80, 0.99, 0.05], [0.85, 0.10, 0.99, 0.05], [0.80, 0.10, 0.95, 0.05]]
P2 = [[0.90, 0.10, 0.05, 0.05], [0.80, 0.20, 0.05, 0.05], [0.10, 0.90, 0.05, 0.05], [0.20, 0.80, 0.05, 0.05]]
P3 = [[0.10, 0.90, 0.99, 0.05], [0.20, 0.80, 0.99, 0.05], [0.90, 0.10, 0.99, 0.05], [0.80, 0.20, 0.99, 0.05]]
# (predictions, max_speakers, chunk_index, expected) -- the reference tests' own vectors
KNOWN = [
    (P1, 2, 0, [(0, 0.0, 0.25), (1, 0.25, 0.5), (0, 0.5, 1.0)]),        # test_two_speaker_cap_keeps_first_arrival_ordered_channels
    (P1, 4, 0, [(0, 0.0, 0.25), (2, 0.25, 1.0)]),                      # test_default_matches_legacy_argmax_across_all_checkpoint_channels
    (P2, 2, 0, [(0, 0.0, 0.5), (1, 0.5, 1.0)]),                        # test_cap_does_not_remap_retained_channel_at_chunk_boundary (first)
    (P3, 2, 1, [(1, 1.0, 1.5), (0, 1.5, 2.0)]),                        #   "  (second chunk, _chunk_index = 1)
]


@pytest.mark.parametrize("preds,cap,chunk,expected", KNOWN)
def test_oracle_reproduces_reference_known_answers(preds, cap, chunk, expected):
    segs, lp = do.process_predictions(np.asarray(preds, np.float32), cap, None, chunk, 1.0, 0.0)
    assert lp == 4
    assert segs == expected


def test_oracle_speaker_cap_rules():
    assert do.resolve_max_speakers(None, 4) == 4                        # sortformer_backend.py:139-140
    assert do.resolve_max_speakers(2, 4) == 2
    for bad in (0, 5, -1, 1.5, True):
        with pytest.raises(ValueError):
            do.resolve_max_speakers(bad, 4)
    with pytest.raises(RuntimeError):                                   # :316-319
        do.frame_segments(np.zeros((3, 2), np.float32), 3, None)
    assert do.process_predictions(np.zeros((0, 4), np.float32), 2, None, 0, 1.0) == ([], 0)


def test_oracle_equals_reference_method_on_random_predictions():
    """The reference's _process_predictions on seeded random cases, recorded by oracle/make_golden_seams.py."""
    from oracle.make_golden_seams import diar_cases
    g = dict(np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "diar_reference.npz")))
    off = g["offsets"]
    for trial, (preds, cap, lp, chunk, gto) in enumerate(diar_cases()):
        sl = slice(off[trial], off[trial + 1])
        ref = [(int(s), float(a), float(b)) for s, a, b in zip(g["speaker"][sl], g["start"][sl], g["end"][sl])]
        mine, my_lp = do.process_predictions(preds, cap, lp, chunk, 0.96, gto)
        assert (mine, my_lp) == (ref, int(g["len_prediction"][trial])), trial


# ------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_device_segments_equal_oracle_bit_exact():
    import torch
    from whisperlivekit_b200.diarization import diar_segments
    rng = np.random.default_rng(11)
    cases = [np.asarray(p, np.float32) for p, *_ in KNOWN]
    for T in (1, 2, 12, 13, 255, 256, 257, 1000, 4096):
        a = rng.random((T, 4)).astype(np.float32)
        if T % 2 == 0:
            a = np.repeat(np.round(a[: max(1, T // 8)], 1), 8, axis=0)[:T]      # runs and ties
        cases.append(a)
    nan = rng.random((20, 4)).astype(np.float32); nan[3, 1] = np.nan; nan[7, 0] = np.nan
    cases.append(nan)
    for cap in (1, 2, 3, 4):
        dev = [torch.from_numpy(c).cuda() for c in cases]
        lps = [max(1, c.shape[0] - (i % 3)) for i, c in enumerate(cases)]          # some streams keep only the tail
        torch.cuda.synchronize()
        got = diar_segments([d.data_ptr() for d in dev], [c.shape[0] for c in cases], lps, 4, cap)
        for i, c in enumerate(cases):
            want, _ = do.frame_segments(c, cap, lps[i])
            assert got[i] == want, (cap, i, c.shape)


@pytest.mark.gpu
def test_segmenter_matches_reference_known_answers_and_errors():
    import torch
    from whisperlivekit_b200 import _lib
    from whisperlivekit_b200.diarization import DiarizationSegmenter, diar_segments
    for preds, cap, chunk, expected in KNOWN:
        s = DiarizationSegmenter(4, 1.0, max_speakers=cap)
        s._chunk_index = chunk
        d = torch.tensor(preds, dtype=torch.float32).cuda()
        torch.cuda.synchronize()
        out = s.process(d.data_ptr(), d.shape[0])
        assert [(x.speaker, x.start, x.end) for x in out] == expected
        assert s._chunk_index == chunk + 1 and s._len_prediction == 4
    # many streams in one call, with silence offsets (insert_silence, sortformer_backend.py:236-245)
    rng = np.random.default_rng(2)
    segs, devs, wants = [], [], []
    for i in range(64):
        s = DiarizationSegmenter(4, 0.96, max_speakers=3)
        s._chunk_index = i
        if i % 5 == 0:
            s.insert_silence(1.37)
        p = rng.random((12, 4)).astype(np.float32)
        segs.append(s); devs.append(torch.from_numpy(p).cuda())
        wants.append(do.process_predictions(p, 3, None, i, 0.96, s.global_time_offset)[0])
    torch.cuda.synchronize()
    out = DiarizationSegmenter.process_batch(segs, [d.data_ptr() for d in devs], [12] * 64)
    assert [[(x.speaker, x.start, x.end) for x in o] for o in out] == wants
    with pytest.raises(_lib.WlkError if hasattr(_lib, "WlkError") else Exception):   # fewer channels than configured (:316-319)
        diar_segments([devs[0].data_ptr()], [12], [12], 2, 3)
