"""CPU: the host logic of bench.py that does not need a GPU -- the real-time paced seam probes (closed cohorts and continuous
batching) over the oracle engine, their summary rule (p95 < chunk period, no backlog growth), and the contract pieces the driver
reads (configs, the reference arm's availability switch)."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from golden_util import case_setup


def test_seam_probes_run_over_the_oracle_engine():
    import bench
    from oracle import whisper_oracle as wo
    g, dims, sd, audio, heads = case_setup("micro")
    eng = wo.OracleEngine(dims, sd, heads)
    eng.max_batch = 8
    rng = np.random.default_rng(0)
    for mode in ("cohort", "continuous"):
        r = bench.seam_probe(eng, 3, 3, 1, rng, mode=mode, context_tokens=20)
        assert r["mode"] == mode and r["errors"] == []
        assert r["engine_calls"] > 0 and r["mean_sessions_per_call"] >= 1.0
        if not r["aborted"]:                                          # the CPU oracle may fall behind real time on a loaded host:
            assert sum(r["stops"].values()) == 3 * 3                  # then the probe gives up (that is its job); otherwise every
            assert 0.0 < r["p50_latency_s"] <= r["p95_latency_s"] <= r["max_latency_s"]   # stream finished every measured tick
        else:
            assert not r["ok"]


def test_seam_summary_rule():
    import bench
    B, ticks, warm = 4, 6, 2
    lat = np.full((B, warm + ticks), 0.2)
    lag = np.full((B, warm + ticks), 0.05)
    stats = dict(prefix=[10], iters=[3], stops={"x": 1})
    ok = bench._seam_summary(B, "cohort", ticks, warm, lat, lag, False, [], stats, 1.0, {})
    assert ok["ok"] and abs(ok["p95_latency_s"] - 0.2) < 1e-9
    slow = lat.copy(); slow[:, -1] = 0.7                                  # p95 over the measured ticks crosses the chunk period
    assert not bench._seam_summary(B, "cohort", ticks, warm, slow, lag, False, [], stats, 1.0, {})["ok"]
    grow = lag.copy(); grow[:, -2:] = 0.4                                 # the start lag grows: a backlog is building
    assert not bench._seam_summary(B, "cohort", ticks, warm, lat, grow, False, [], stats, 1.0, {})["ok"]
    assert not bench._seam_summary(B, "cohort", ticks, warm, lat, lag, True, [], stats, 1.0, {})["ok"]
    assert not bench._seam_summary(B, "cohort", ticks, warm, lat, lag, False, ["boom"], stats, 1.0, {})["ok"]


def test_contract_pieces():
    import bench
    assert bench.CONFIGS[0] == "alignatt-large-v3" and len(bench.CONFIGS) == 6
    assert bench.CHUNK == 8000 and bench.WINDOW == 480000 and bench.CHUNK_S == 0.5
    peaks = bench.load_peaks()
    assert peaks["bf16_tflops"] > 100 and peaks["hbm_gbs"] > 1000
    assert isinstance(bench.reference_available(), bool)


def test_dump_outputs_writes_float_arrays_within_the_limit(tmp_path):
    import bench
    out = dict(tokens=np.arange(6, dtype=np.float64).reshape(2, 3), logprobs=np.full(3, -0.5, np.float32))
    bench.dump_outputs(str(tmp_path / "d"), out)
    for name, a in out.items():
        got = np.load(tmp_path / "d" / f"{name}.npy")
        assert got.dtype == a.dtype and np.array_equal(got, a)
    with pytest.raises(ValueError):
        bench.dump_outputs(str(tmp_path / "big"), dict(x=np.zeros(9, np.float64)), limit=64)
    assert not (tmp_path / "big").exists()


def test_scripted_tick_records_what_it_returned():
    """bench.scripted_tick over the oracle engine: --dump-outputs (scripted_tick_outputs) holds exactly what the tick's
    engine calls returned, and the logits its last decode left, against the same calls made directly."""
    import bench
    from oracle import whisper_oracle as wo
    g, dims, sd, audio, heads = case_setup("micro")
    engines = [wo.OracleEngine(dims, sd, heads) for _ in range(2)]
    sids = [[e.open_session() for _ in range(2)] for e in engines]
    for e, ss in zip(engines, sids):
        for k, s in enumerate(ss):
            e.append_audio(s, audio[k * 8000:])
    sp = engines[0].specials
    prefix = list(sp.sot_sequence_including_notimestamps()) + [1169, 2068]
    sup = sp.alignatt_suppress_tokens()
    host = dict(encode=0.0, prefill=0.0, prefill_synced=0.0, step=0.0, n=0, ns=0)
    last = {}
    bench.scripted_tick(engines[0], sids[0], prefix, sup, host, last)
    got = bench.scripted_tick_outputs(engines[0], sids[0], last, logits_bytes=4 * dims.n_vocab)
    assert host["n"] == 1 and set(got) == {"content_frames", "no_speech_prob", "tokens", "logprobs", "frames", "logits"}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())

    e, ss = engines[1], sids[1]                                           # the same calls, made directly
    assert got["content_frames"].tolist() == e.encode(ss)
    e.decode(ss, [prefix] * len(ss))
    np.testing.assert_array_equal(got["no_speech_prob"], np.asarray(e.no_speech_prob(ss), np.float32))
    assert got["tokens"].shape == (bench.STEPS_PER_CHUNK, len(ss))
    for it in range(bench.STEPS_PER_CHUNK):
        r = e.select(ss, sup)
        assert got["tokens"][it].tolist() == [t for t, _, _ in r] and got["frames"][it].tolist() == [f for _, _, f in r]
        np.testing.assert_array_equal(got["logprobs"][it], np.asarray([p for _, p, _ in r], np.float32))
        e.decode(ss, [[t] for t, _, _ in r])
    assert got["logits"].shape == (1, dims.n_vocab)                       # the cap keeps the first session's row
    np.testing.assert_array_equal(got["logits"][0], e.read_logits(ss[0]))
