"""Needs the reference package staged under oracle/_ref by build(): the drop-in seam.  The reference's own
AlignAttBase.infer() drives our hooks (AlignAttHooks); with the CPU oracle standing in for the
CUDA engine behind the same session API, the emitted tokens / attended frames must equal what the
reference's AlignAtt produced (the golden fixtures)."""
import numpy as np
import pytest
import torch

from golden_util import case_setup

pytestmark = pytest.mark.reference


@pytest.fixture(autouse=True)
def _reference_on_the_cpu(monkeypatch):
    """The reference puts AlignAtt on the GPU whenever one is visible; here it runs next to the CPU oracle."""
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)


def _import_reference():
    from oracle import stage_reference
    stage_reference.import_staged_reference()


@pytest.mark.parametrize("name", ["micro", "microml"])
@pytest.mark.parametrize("tag,nsp", [("pol", 1.01), ("poldef", 0.5)])
def test_reference_infer_over_b200_hooks(name, tag, nsp):
    _import_reference()
    from oracle import whisper_oracle as wo
    from whisperlivekit.simul_whisper.config import AlignAttConfig as RefCfg
    from whisperlivekit_b200.plugin import B200WhisperModel, make_b200_alignatt_class

    g, dims, sd, audio, heads = case_setup(name)
    model = B200WhisperModel(wo.OracleEngine(dims, sd, heads))
    cfg = RefCfg(tokenizer_is_multilingual=dims.is_multilingual, language="en", audio_min_len=0.0, audio_max_len=30.0,
                 decoder_type="greedy", beam_size=1, segment_length=0.5, frame_threshold=25, nonspeech_prob=nsp)
    a = make_b200_alignatt_class()(cfg=cfg, loaded_model=model)
    frames_log, toks_log = [], []
    of, ou = a._get_attended_frames, a._update_tokens
    a._get_attended_frames = lambda attn: (lambda r: (frames_log.append(r[1]), r)[1])(of(attn))
    a._update_tokens = lambda ct, lg, sl: (lambda r: (toks_log.append(int(r[0][0, -1])), r)[1])(ou(ct, lg, sl))
    new_tokens, step_tokens, step_frames = [], [], []
    n_chunks = int(np.ceil(len(audio) / 8000))
    for c in range(n_chunks):
        a.insert_audio(torch.from_numpy(audio[c * 8000:(c + 1) * 8000]))
        frames_log.clear(); toks_log.clear()
        n_before = len(a.state.tokens)
        words = a.infer(is_last=(c == n_chunks - 1))
        assert isinstance(words, list)
        if len(a.state.tokens) > n_before:
            new_tokens += a.state.tokens[-1][0].tolist()
        step_tokens += list(toks_log); step_frames += list(frames_log)
    assert step_tokens == list(g[f"{tag}_step_tokens"])
    assert step_frames == list(g[f"{tag}_step_frames"])
    assert new_tokens == list(g[f"{tag}_new_tokens"])


@pytest.mark.parametrize("name,beam", [("micro", 3), ("microml", 2)])
def test_reference_beam_search_over_forked_sessions(name, beam):
    """decoder_type="beam": the reference's AlignAtt (BeamPyTorchInference + BeamSearchDecoder over its torch
    Whisper, simul_whisper.py:182-192) and the reference's infer() over our hooks -- beam rows as forked sessions,
    rearrange_kv_cache as gather_decoder -- run side by side on the same stream and must agree step by step."""
    _import_reference()
    from oracle import whisper_oracle as wo
    from oracle.make_golden import build_reference_model
    from whisperlivekit.simul_whisper.config import AlignAttConfig as RefCfg
    from whisperlivekit.simul_whisper.simul_whisper import AlignAtt
    from whisperlivekit_b200.plugin import B200WhisperModel, make_b200_alignatt_class

    g, dims, sd, audio, heads = case_setup(name)

    def cfg():
        return RefCfg(tokenizer_is_multilingual=dims.is_multilingual, language="en", audio_min_len=0.0,
                      audio_max_len=30.0, decoder_type="beam", beam_size=beam, segment_length=0.5, frame_threshold=25,
                      nonspeech_prob=1.01)

    ref = AlignAtt(cfg=cfg(), loaded_model=build_reference_model(dims, sd, heads))
    eng = wo.OracleEngine(dims, sd, heads)
    mine = make_b200_alignatt_class()(cfg=cfg(), loaded_model=B200WhisperModel(eng))
    assert len(mine.beam_sids) == beam
    gathers = []
    og = eng.gather_decoder
    eng.gather_decoder = lambda sids, src: (gathers.append(list(src)), og(sids, src))[1]

    logs = {}
    for tag, a in (("ref", ref), ("mine", mine)):
        logs[tag] = dict(frames=[], toks=[])

        def spy_frames(attn, _o=a._get_attended_frames, _l=logs[tag]["frames"]):
            r = _o(attn); _l.append(([int(x) for x in r[0]], int(r[1]))); return r

        def spy_update(ct, lg, sl, _o=a._update_tokens, _l=logs[tag]["toks"]):
            r = _o(ct, lg, sl); _l.append((r[0].tolist(), bool(r[1]))); return r

        a._get_attended_frames, a._update_tokens = spy_frames, spy_update

    n_chunks = int(np.ceil(len(audio) / 8000))
    n_steps = 0
    for c in range(n_chunks):
        seg = torch.from_numpy(audio[c * 8000:(c + 1) * 8000])
        ref.insert_audio(seg); mine.insert_audio(seg.clone())
        for l in logs.values():
            l["frames"].clear(); l["toks"].clear()
        wr = ref.infer(is_last=(c == n_chunks - 1))
        wm = mine.infer(is_last=(c == n_chunks - 1))
        assert logs["mine"]["toks"] == logs["ref"]["toks"], f"chunk {c}: beam candidates diverged"
        assert logs["mine"]["frames"] == logs["ref"]["frames"], f"chunk {c}: attended frames diverged"
        assert [(w.text, w.start, w.end) for w in wm] == [(w.text, w.start, w.end) for w in wr]
        assert [t.tolist() for t in mine.state.tokens] == [t.tolist() for t in ref.state.tokens]
        n_steps += len(logs["ref"]["toks"])
    assert n_steps > 20                                  # the beams really decoded
    assert any(src != list(range(beam)) for src in gathers)      # and the K/V rows really were re-indexed
