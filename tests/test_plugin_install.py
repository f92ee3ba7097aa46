"""Needs the reference package staged under oracle/_ref by build(): ``plugin.install()`` executed against the
reference's own ``SimulStreamingASR`` / ``SimulStreamingOnlineProcessor`` (simul_whisper/backend.py:61-71, 530-553),
and the two hooks no other test reaches -- ``lang_id`` (simul_whisper.py:266-292) and the CIF end-of-word test
(eow_detection.py:37-77).  The CUDA engine is replaced by the CPU oracle through ``install(engine_factory=...)``:
what is under test is the registration and the hooks, not the kernels (those are the -m gpu tests)."""
import os
import types

import numpy as np
import pytest
import torch

from golden_util import case_setup


@pytest.fixture(autouse=True)
def _reference_on_the_cpu(monkeypatch):
    """The reference puts AlignAtt on the GPU whenever one is visible; here it runs next to the CPU oracle."""
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)


def _import_reference():
    from oracle import stage_reference
    stage_reference.import_staged_reference()


ASR_KW = dict(decoder_type="greedy", beams=1, model_size=None, model_path=None, decoder_model_path=None,
              encoder_model_path=None, backend="whisper", min_chunk_size=0.5, frame_threshold=25, lan="en",
              audio_max_len=30.0, audio_min_len=0.0, cif_ckpt_path=None, direct_english_translation=False,
              never_fire=False, init_prompt=None, max_context_tokens=None, static_init_prompt=None, warmup_file=False,
              custom_alignment_heads=None, model_cache_dir=None, lora_path=None, disable_fast_encoder=True)


def _checkpoint(tmp_path, name, dims, sd, heads):
    """A Whisper ``.pt`` as the reference's load_model reads it (whisper/__init__.py:516-596)."""
    ck = {"dims": dict(zip(["n_mels", "n_audio_ctx", "n_audio_state", "n_audio_head", "n_audio_layer", "n_vocab", "n_text_ctx",
                            "n_text_state", "n_text_head", "n_text_layer"], dims.as_tuple())),
          "model_state_dict": {k: torch.from_numpy(v) for k, v in sd.items()}}
    path = os.path.join(tmp_path, name)
    torch.save(ck, path)
    return path


@pytest.mark.reference
def test_install_routes_simulstreaming_through_the_engine(tmp_path, monkeypatch):
    _import_reference()
    import whisperlivekit.simul_whisper.backend as be
    monkeypatch.setattr(be, "load_file", lambda *a, **k: None)      # warm-up file loader needs librosa (absent here)
    from oracle import whisper_oracle as wo
    from oracle.make_golden import build_reference_model
    from whisperlivekit.simul_whisper.simul_whisper import AlignAtt as RefAlignAtt
    from whisperlivekit_b200 import plugin
    from whisperlivekit_b200.weights import state_dict_from_torch

    g, dims, sd, audio, heads = case_setup("micro")
    name = "micro.en.pt" if not dims.is_multilingual else "micro.pt"
    path = _checkpoint(str(tmp_path), name, dims, sd, heads)
    seen = {}

    def factory(torch_model):
        seen["dims"] = torch_model.dims
        return wo.OracleEngine(dims, state_dict_from_torch(torch_model.state_dict()), heads)

    def run(install):
        if install:
            cls = plugin.install(batching=True, max_batch=4, engine_factory=factory)
            assert be.AlignAtt is cls
        else:
            plugin.uninstall()
            assert be.AlignAtt is RefAlignAtt
        kw = dict(ASR_KW, model_path=path)
        asr = be.SimulStreamingASR(**kw)
        if not install:                                  # the reference's own model needs the alignment heads we test with
            mask = torch.zeros(dims.n_text_layer, dims.n_text_head, dtype=torch.bool)
            for l, h in heads:
                mask[l, h] = True
            asr.shared_model.register_buffer("alignment_heads", mask.to_sparse(), persistent=False)
        asr.cfg.nonspeech_prob = 1.01
        proc = be.SimulStreamingOnlineProcessor(asr)
        toks = []
        n_chunks = int(np.ceil(len(audio) / 8000))
        for c in range(n_chunks):
            proc.insert_audio_chunk(audio[c * 8000:(c + 1) * 8000], (c + 1) * 0.5)
            proc.process_iter(is_last=(c == n_chunks - 1))
            toks.append([t[0].tolist() for t in proc.model.state.tokens[1:]])
        return asr, proc, toks

    try:
        asr, proc, toks_b200 = run(True)
        assert type(proc.model).__name__ == "B200AlignAtt"
        assert type(asr.shared_model).__name__ == "B200WhisperModel"
        assert seen["dims"].n_audio_state == dims.n_audio_state
        eng = asr.shared_model.engine                      # BatchingEngine over the factory's engine
        assert eng.stats["calls"] > 0
        sid = proc.model.sid
        proc.__del__()                                     # teardown releases the session (plugin.processor_del)
        with pytest.raises(Exception):
            eng.engine.audio_len(sid)
        eng.close()
    finally:
        plugin.uninstall()
    # the same stream through the unmodified reference: same hypothesis tokens, chunk by chunk
    asr_ref, proc_ref, toks_ref = run(False)
    assert type(proc_ref.model) is RefAlignAtt
    assert toks_b200 == toks_ref


@pytest.mark.reference
def test_lang_id_hook_matches_reference():
    _import_reference()
    from oracle import whisper_oracle as wo
    from oracle.make_golden import build_reference_model
    from whisperlivekit.simul_whisper.config import AlignAttConfig as RefCfg
    from whisperlivekit.simul_whisper.simul_whisper import AlignAtt
    from whisperlivekit_b200.plugin import B200WhisperModel, make_b200_alignatt_class

    g, dims, sd, audio, heads = case_setup("microml")
    assert dims.is_multilingual

    def cfg():
        return RefCfg(tokenizer_is_multilingual=True, language="auto", audio_min_len=0.0, audio_max_len=30.0,
                      decoder_type="greedy", beam_size=1, segment_length=0.5, frame_threshold=25)

    ref = AlignAtt(cfg=cfg(), loaded_model=build_reference_model(dims, sd, heads))
    ours = make_b200_alignatt_class()(cfg=cfg(), loaded_model=B200WhisperModel(wo.OracleEngine(dims, sd, heads)))
    seg = torch.from_numpy(audio[:48000])
    ref.insert_audio(seg); ours.insert_audio(seg)
    with torch.no_grad():
        enc_r, _ = ref._encode(ref._concat_segments())
        t_r, p_r = ref.lang_id(enc_r)
    enc_o, _ = ours._encode(ours._concat_segments())
    t_o, p_o = ours.lang_id(enc_o)
    assert int(t_r[0]) == int(t_o[0])
    assert set(p_r[0]) == set(p_o[0])
    top_r = max(p_r[0].items(), key=lambda x: x[1])
    top_o = max(p_o[0].items(), key=lambda x: x[1])
    assert top_r[0] == top_o[0]                                           # what infer() consumes (align_att_base.py:162)
    assert max(abs(p_r[0][c] - p_o[0][c]) for c in p_r[0]) < 1e-5
    # the decoder state is clean afterwards: a normal infer() follows (align_att_base.py:164-170 re-inits tokens)
    ours.create_tokenizer(top_o[0]); ours.init_tokens(); ours.init_context()
    assert isinstance(ours.infer(is_last=False), list)


@pytest.mark.reference
def test_cif_fire_at_boundary_matches_reference(tmp_path):
    _import_reference()
    from oracle import whisper_oracle as wo
    from oracle.make_golden import build_reference_model
    from whisperlivekit.simul_whisper.config import AlignAttConfig as RefCfg
    from whisperlivekit.simul_whisper.simul_whisper import AlignAtt
    from whisperlivekit_b200.plugin import B200WhisperModel, make_b200_alignatt_class

    g, dims, sd, audio, heads = case_setup("micro")
    torch.manual_seed(5)
    lin = torch.nn.Linear(dims.n_audio_state, 1)
    ck = os.path.join(str(tmp_path), "cif.pt")
    torch.save(lin.state_dict(), ck)

    def cfg():
        return RefCfg(tokenizer_is_multilingual=dims.is_multilingual, language="en", audio_min_len=0.0, audio_max_len=30.0,
                      decoder_type="greedy", beam_size=1, segment_length=0.5, frame_threshold=25, cif_ckpt_path=ck)

    ref = AlignAtt(cfg=cfg(), loaded_model=build_reference_model(dims, sd, heads))
    ours = make_b200_alignatt_class()(cfg=cfg(), loaded_model=B200WhisperModel(wo.OracleEngine(dims, sd, heads)))
    assert ours.state.CIFLinear is not None and not ours.state.always_fire
    fired = []
    for n in (16000, 40000, 72000, len(audio)):
        for a in (ref, ours):
            a.refresh_segment(complete=True)
            a.insert_audio(torch.from_numpy(audio[:n]))
        with torch.no_grad():
            enc_r, c_r = ref._encode(ref._concat_segments())
            f_r = bool(ref.fire_at_boundary(enc_r[:, :c_r, :]))
        enc_o, c_o = ours._encode(ours._concat_segments())
        f_o = bool(ours.fire_at_boundary(enc_o[:, :c_o, :]))
        assert c_r == c_o
        assert f_r == f_o
        fired.append(f_r)
    # and through the whole infer(): the CIF decision only changes how many tokens are kept (align_att_base.py:296)
    assert isinstance(ours.infer(is_last=False), list)


@pytest.mark.reference
def test_reference_diarization_factory_builds_the_sortformer_drop_in():
    """plugin.install_sortformer() + the reference's unchanged core.online_diarization_factory (core.py:468-480): its own
    import statement resolves to the B200 drop-in and its calling convention constructs it.  The shared model carries
    only what that constructor reads; the drop-ins run end to end on the GPU in
    tests/test_gpu_sortformer.py::test_registration_as_the_reference_backend_module."""
    _import_reference()
    from whisperlivekit_b200 import plugin
    from whisperlivekit_b200.sortformer_dims import SORTFORMER_DIMS
    from whisperlivekit_b200.sortformer_engine import B200SortformerDiarizationOnline
    d = SORTFORMER_DIMS["small"]
    mod = plugin.install_sortformer(dims=d)
    try:
        from whisperlivekit.core import online_diarization_factory
        opened = []
        engine = types.SimpleNamespace(chunk_duration_seconds=1.0, device=0, open_session=lambda: opened.append(7) or 7)
        args = types.SimpleNamespace(diarization_backend="sortformer", sortformer_max_speakers=2)
        online = online_diarization_factory(args, types.SimpleNamespace(engine=engine, dims=d))
        assert type(online) is mod.SortformerDiarizationOnline is B200SortformerDiarizationOnline
        assert online.engine is engine and online.sid == 7 and opened == [7] and online.max_speakers == 2
    finally:
        plugin.uninstall_sortformer()


def test_nemo_checkpoint_reader_needs_no_nemo(tmp_path):
    """plugin.sortformer_state_dict_from_nemo: a .nemo file is a tar holding model_weights.ckpt (a torch state_dict under NeMo's
    parameter names); the reader returns numpy arrays and the engine-side loader skips the buffers of modules this path
    replaces (checked on the GPU in tests/test_gpu_sortformer.py)."""
    import io
    import tarfile

    import numpy as np
    import torch

    from whisperlivekit_b200 import plugin
    from whisperlivekit_b200.sortformer_dims import SORTFORMER_DIMS, synthetic_sortformer_state_dict
    d = SORTFORMER_DIMS["micro"]
    sd = synthetic_sortformer_state_dict(d, 3)
    blob = io.BytesIO()
    torch.save({k: torch.from_numpy(v) for k, v in sd.items()}, blob)
    path = tmp_path / "diar_streaming_sortformer_4spk-v2.nemo"
    with tarfile.open(path, "w") as tar:
        for name, data in (("./model_config.yaml", b"name: sortformer\n"), ("./model_weights.ckpt", blob.getvalue())):
            info = tarfile.TarInfo(name)
            info.size = len(data)
            tar.addfile(info, io.BytesIO(data))
    got = plugin.sortformer_state_dict_from_nemo(str(path))
    assert sorted(got) == sorted(sd)
    for k in sd:
        assert got[k].dtype == np.float32 and np.array_equal(got[k], sd[k])
