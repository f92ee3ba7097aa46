"""CPU: the oracle restatement against fixtures recorded from the real reference
(oracle/make_golden.py), plus host-logic checks.  Tolerances: fp32 CPU vs fp32
CPU of the same algorithm -> 2e-4 abs on O(1..10) tensors; integer traces exact."""
import numpy as np
import pytest
import torch

from golden_util import case_setup, load_case, run_policy, sampled_diff, GOLDEN
from oracle import whisper_oracle as wo
from whisperlivekit_b200.dims import DIMS, SpecialTokens, ALIGNMENT_HEADS
from whisperlivekit_b200.weights import mel_filterbank

CASES = ["micro", "microml", "tiny"]


def test_mel_filterbank_matches_reference_asset():
    g = dict(np.load(f"{GOLDEN}/mel_filters.npz"))
    for n in (80, 128):
        mine = mel_filterbank(n)
        assert float(g[f"max_abs_diff_{n}"]) < 1e-8
        np.testing.assert_allclose(mine.reshape(-1)[g[f"idx_{n}"]], g[f"val_{n}"], atol=1e-8, rtol=0)
        np.testing.assert_allclose(mine.sum(1), g[f"rowsum_{n}"], atol=1e-7, rtol=0)


@pytest.mark.parametrize("name", CASES)
def test_special_tokens_match_reference_tokenizer(name):
    g, dims, *_ = case_setup(name)
    sp = SpecialTokens.for_dims(dims)
    assert list(g["blank_token"]) == [sp.blank]
    assert list(g["suppress_tokens"]) == sp.alignatt_suppress_tokens()
    assert list(g["initial_tokens"]) == list(sp.sot_sequence_including_notimestamps())


@pytest.mark.parametrize("name", CASES)
def test_oracle_tensors_match_reference(name):
    g, dims, sd, audio, heads = case_setup(name)
    W = wo.Weights(sd)
    with torch.no_grad():
        mel, content = wo.encode_features(torch.from_numpy(audio), mel_filterbank(dims.n_mels))
        assert content == int(g["content_mel_len"])
        d, m = sampled_diff(g, "mel", mel[0].numpy())
        assert d < 2e-5, d
        enc = wo.encoder_forward(W, dims, mel)
        d, m = sampled_diff(g, "enc", enc[0].numpy())
        assert d < 2e-4, (d, m)
        kv = {}
        prefix = torch.tensor([list(g["forced_prefix"])])
        logits, cross = wo.decoder_forward(W, dims, prefix, enc, kv)
        assert sampled_diff(g, "logits_prefill_last", logits[0, -1].numpy())[0] < 3e-4
        assert sampled_diff(g, "logits_prefill_sot", logits[0, 0].numpy())[0] < 3e-4
        assert list(logits[0].argmax(-1).numpy()) == list(g["argmax_prefill"])
        acc, am = [cross], []
        for i, t in enumerate(g["forced_steps"]):
            logits, cross = wo.decoder_forward(W, dims, torch.tensor([[int(t)]]), enc, kv)
            acc.append(cross)
            am.append(int(logits[0, -1].argmax()))
            if i in (0, 4):
                assert sampled_diff(g, f"logits_step{i}", logits[0, -1].numpy())[0] < 3e-4
        assert am == list(g["argmax_steps"])
        attn = wo.process_cross_attention(acc, heads, dims.n_text_layer, content)
        assert sampled_diff(g, "align_attn", attn[0].numpy())[0] < 2e-3
        assert list(attn[0].argmax(-1).numpy()) == list(g["align_argmax_rows"])


@pytest.mark.parametrize("name", ["micro", "microml"])
@pytest.mark.parametrize("tag,nsp", [("pol", 1.01), ("poldef", 0.5)])
def test_policy_on_oracle_matches_reference_alignatt(name, tag, nsp):
    """StreamingAlignAtt (host mirror) + OracleEngine == reference AlignAtt.infer."""
    g, dims, sd, audio, heads = case_setup(name)
    eng = wo.OracleEngine(dims, sd, heads)
    tr = run_policy(eng, audio, nsp)
    for k in ("step_tokens", "step_frames", "step_offsets", "new_tokens", "new_tokens_offsets"):
        assert list(tr[k]) == list(g[f"{tag}_{k}"]), k


def test_alignment_heads_table_shape():
    for k, heads in ALIGNMENT_HEADS.items():
        d = DIMS[k]
        assert all(0 <= l < d.n_text_layer and 0 <= h < d.n_text_head for l, h in heads)
        assert heads == sorted(heads)


def test_alignment_heads_match_reference():
    """The reference's _ALIGNMENT_HEADS table, decoded (oracle/make_golden_seams.py)."""
    g = load_case("alignment_heads")
    for k, heads in ALIGNMENT_HEADS.items():
        d = DIMS[k]
        a = g[k]
        assert a.shape == (d.n_text_layer, d.n_text_head)
        assert [(int(l), int(h)) for l, h in zip(*np.nonzero(a))] == heads
