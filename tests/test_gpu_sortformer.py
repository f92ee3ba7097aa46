"""GPU: the streaming Sortformer engine (wlk_sf_*, through the C ABI) against the CPU oracle (oracle/sortformer_oracle.py --
a restatement of NeMo's algorithm, PARITY UNPINNED) on seeded weights: chunk predictions, speaker cache / FIFO / silence
profile after every step (several cache compressions inside), ragged batches, the feature-level seam, and the segments
of the device post-processing against the reference-pinned oracle of `_process_predictions`."""
import asyncio
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _setup(name, seed):
    from oracle.sortformer_oracle import SortformerOracle
    from whisperlivekit_b200.sortformer_dims import SORTFORMER_DIMS, synthetic_sortformer_state_dict
    d = SORTFORMER_DIMS[name]
    sd = synthetic_sortformer_state_dict(d, seed)
    return d, sd, SortformerOracle(d, sd)


def _compare_state(eng, sid, st, tol):
    s = eng.read_state(sid)
    assert s["spkcache_len"] == st["spkcache_len"] and s["fifo_len"] == st["fifo_len"]
    assert s["n_sil"] == st["n_sil"]
    sl, fl = st["spkcache_len"], st["fifo_len"]
    assert np.abs(s["fifo"][:fl] - st["fifo"][:fl].numpy()).max(initial=0.0) < tol
    assert np.abs(s["mean_sil_emb"] - st["mean_sil_emb"].numpy()).max() < tol
    assert np.abs(s["spkcache"][:sl] - st["spkcache"][:sl].numpy()).max(initial=0.0) < tol
    assert np.abs(s["spkcache_preds"][:sl] - st["spkcache_preds"][:sl].numpy()).max(initial=0.0) < tol


@pytest.mark.parametrize("name,steps", [("micro", 12), ("small", 9)])
def test_fp32_engine_matches_oracle_over_a_stream(name, steps):
    from oracle.sortformer_oracle import OracleDiarizer
    from whisperlivekit_b200.sortformer_dims import synthetic_two_speaker_audio
    from whisperlivekit_b200.sortformer_engine import SortformerEngine
    d, sd, model = _setup(name, 7)
    eng = SortformerEngine(d, sd, precision="fp32", max_sessions=2, max_batch=2)
    sid = eng.open_session()
    orc = OracleDiarizer(model)
    audio = synthetic_two_speaker_audio(steps + 1.0, seed=21)
    worst = 0.0
    for k in range(steps):
        chunk = audio[k * 16000:(k + 1) * 16000]
        want = orc.step(chunk).numpy()
        got = eng.step_audio([sid], [chunk])[0]
        assert got.shape == want.shape
        worst = max(worst, float(np.abs(got - want).max()))
        assert worst < 1e-3, (k, worst)                     # sigmoid outputs in (0, 1): north_star's 1e-3
        _compare_state(eng, sid, orc.st, 2e-3)
    assert orc.st["spkcache_len"] == d.spkcache_len          # the stream was long enough to compress the cache
    eng.close()


def test_fp32_ragged_batch_and_feature_seam():
    """Streams that started at different times share calls; one stream is driven through the forward_streaming_step seam
    (features in) and must equal the audio path."""
    from oracle.sortformer_oracle import OracleDiarizer, log_mel
    from whisperlivekit_b200.sortformer_dims import synthetic_two_speaker_audio
    from whisperlivekit_b200.sortformer_engine import SortformerEngine
    import torch
    d, sd, model = _setup("small", 11)
    eng = SortformerEngine(d, sd, precision="fp32", max_sessions=4, max_batch=4)
    audios = [synthetic_two_speaker_audio(9.0, seed=40 + i) * (0.4 + 0.2 * i) for i in range(3)]
    sids = [eng.open_session() for _ in range(3)]
    orcs = [OracleDiarizer(model) for _ in range(3)]
    feat_sid = eng.open_session()
    prev = None
    start = [0, 2, 3]                                        # stream i joins at call start[i]
    for call in range(8):
        live = [i for i in range(3) if call >= start[i]]
        chunks = [audios[i][(call - start[i]) * 16000:(call - start[i] + 1) * 16000] for i in live]
        got = eng.step_audio([sids[i] for i in live], chunks)
        for i, g, c in zip(live, got, chunks):
            want = orcs[i].step(c).numpy()
            assert g.shape == want.shape and np.abs(g - want).max() < 1e-3, (call, i)
        # stream 0 again, through the feature seam (the reference's own mel + 99-frame overlap, sortformer_backend.py:273-287)
        mel = log_mel(chunks[0], d)
        total = mel if prev is None else torch.cat([prev[:, -99:], mel], dim=1)
        prev = mel
        f = eng.step_features([feat_sid], [total.t().contiguous().numpy()], 8 if call > 0 else 0, 8)[0]
        assert np.abs(f - got[0]).max() < 1e-3, call
    for i in range(3):
        _compare_state(eng, sids[i], orcs[i].st, 2e-3)
    eng.close()


def test_error_contract():
    from whisperlivekit_b200 import _lib
    from whisperlivekit_b200.sortformer_engine import SortformerEngine
    d, sd, _ = _setup("micro", 1)
    eng = SortformerEngine(d, sd, precision="fp32", max_sessions=2, max_batch=2)
    s = eng.open_session()
    with pytest.raises(_lib.WlkError, match="exactly"):
        eng.step_audio([s], [np.zeros(15999, np.float32)])
    with pytest.raises(_lib.WlkError, match="twice"):
        eng.step_audio([s, s], [np.zeros(16000, np.float32)] * 2)
    with pytest.raises(_lib.WlkError, match="invalid session"):
        eng.step_audio([1], [np.zeros(16000, np.float32)])
    st = eng.read_state(s)
    assert st["chunk_index"] == 0 and st["fifo_len"] == 0     # failed calls left the session untouched
    eng.step_audio([s], [np.zeros(16000, np.float32)])
    eng.reset_session(s)
    assert eng.read_state(s)["chunk_index"] == 0
    eng.close()


def test_bf16_true_geometry_tracks_oracle_and_seam_objects():
    """The 17 x 512 / 18 x 192 geometry in the serving mode (bf16 tcgen05 GEMMs) against the fp32 oracle, through the
    drop-in objects of the diarization seam; segments = the reference-pinned post-processing of the oracle's predictions
    wherever the oracle's top-2 margin exceeds the bf16 error."""
    from oracle.diar_oracle import frame_segments
    from oracle.sortformer_oracle import OracleDiarizer, SortformerOracle
    from whisperlivekit_b200.sortformer_dims import SORTFORMER_DIMS, synthetic_sortformer_state_dict, synthetic_two_speaker_audio
    from whisperlivekit_b200.sortformer_engine import B200SortformerDiarization, B200SortformerDiarizationOnline
    d = SORTFORMER_DIMS["diar_streaming_sortformer_4spk-v2"]
    sd = synthetic_sortformer_state_dict(d, 3)
    shared = B200SortformerDiarization(d, sd, precision="bf16", max_sessions=2, max_batch=2)
    online = B200SortformerDiarizationOnline(shared, max_speakers=3)
    assert hasattr(online, "buffer_audio") and online.chunk_duration_seconds == 1.0
    orc = OracleDiarizer(SortformerOracle(d, sd))
    audio = synthetic_two_speaker_audio(4.0, seed=9)
    worst = 0.0
    for k in range(8):                                       # 0.5 s pieces: diarize() fires every second one
        online.insert_audio_chunk(audio[k * 8000:(k + 1) * 8000])
        segs = asyncio.run(online.diarize())
        if k % 2 == 0:
            assert segs == []
            continue
        want = orc.step(audio[(k // 2) * 16000:(k // 2 + 1) * 16000]).numpy()
        ptr, rows = shared.engine.total_preds(online.sid)
        assert rows == orc.total_preds.shape[0]
        s = shared.engine.read_state(online.sid)
        assert s["fifo_len"] == orc.st["fifo_len"]
        got_all = _read_device(ptr, rows * d.n_spk).reshape(rows, d.n_spk)     # device -> host through torch (plumbing only)
        got_tail = got_all[-want.shape[0]:]
        worst = max(worst, float(np.abs(got_tail - want).max()))
        lp = 12
        ref_segs, _ = frame_segments(orc.total_preds.numpy(), 3, lp)
        top2 = np.sort(orc.total_preds.numpy()[-lp:, :3], axis=1)
        if (top2[:, -1] - top2[:, -2]).min() > 2 * worst + 1e-3:
            assert [(s_.speaker) for s_ in segs] == [a for a, _, _ in ref_segs]
    assert worst < 6e-2, worst
    online.close()
    shared.close()


def test_registration_as_the_reference_backend_module():
    """plugin.install_sortformer(): the module the reference's core.online_diarization_factory (core.py:468-480) imports
    holds the B200 drop-ins although NeMo is absent (the real module would exit at import), a checkpoint-shaped state_dict
    with NeMo's extra buffers loads, and drop-ins built with the factory's keyword arguments serve audio_processor's calls
    end to end.  That the factory itself resolves to these classes is checked where the reference package is staged
    (tests/test_plugin_install.py::test_reference_diarization_factory_builds_the_sortformer_drop_in)."""
    from whisperlivekit_b200 import plugin
    from whisperlivekit_b200.sortformer_dims import SORTFORMER_DIMS, synthetic_sortformer_state_dict, synthetic_two_speaker_audio
    d = SORTFORMER_DIMS["small"]
    sd = dict(synthetic_sortformer_state_dict(d, 2))
    sd["preprocessor.featurizer.window"] = np.zeros(400, np.float32)                  # buffers a .nemo state_dict also holds
    sd["encoder.layers.0.conv.batch_norm.num_batches_tracked"] = np.asarray(7, np.int64)
    sd["sortformer_modules.hidden_to_spks.weight"] = np.zeros((d.n_spk, 2 * d.tf_d_model), np.float32)
    plugin.install_sortformer(state_dict=sd, dims=d, precision="fp32", max_sessions=2, max_batch=2)
    try:
        backend = sys.modules["whisperlivekit.diarization.sortformer_backend"]
        shared = backend.SortformerDiarization(model_path=None)
        online = backend.SortformerDiarizationOnline(shared_model=shared, max_speakers=2)      # as the factory builds it
        assert hasattr(online, "buffer_audio") and online.max_speakers == 2
        audio = synthetic_two_speaker_audio(2.5, seed=4)
        got = []
        for k in range(5):
            online.insert_audio_chunk(audio[k * 8000:(k + 1) * 8000])
            got.append(asyncio.run(online.diarize()))
        assert got[0] == [] and got[2] == [] and len(got[1]) >= 1 and len(got[3]) >= 1
        assert got[1][0].start == 0.0 and got[3][-1].end == 2.0 and all(0 <= s.speaker < 2 for s in got[1] + got[3])
        online.insert_silence(1.5)
        online.close(); shared.close()
    finally:
        plugin.uninstall_sortformer()


def _read_device(ptr, n):
    import torch

    class _Blob:
        __cuda_array_interface__ = dict(shape=(n,), typestr="<f4", data=(ptr, False), version=2)
    return torch.as_tensor(_Blob(), device="cuda").cpu().numpy().copy()
