"""Op-level checks of the decoder attention kernels through wlk_op_decoder_attention, against plain torch fp64
references on the inputs the kernels saw (bf16-rounded where they read bf16).

The op runs the dispatch of wlk_decode: the SIMT kernels (dec_self_attn_kernel / dec_cross_attn_kernel with one or
eight queries per pass) and, on the tensor-core backend, attn_tc_kernel in MODE_SELF / MODE_CROSS with the SIMT kernel
exporting the alignment heads' rows.

Two kinds of input:
  * structured probes, built so that a wrong index moves the output by O(1) whatever the tolerance: V carries each
    key's position split over two dims (bf16(p) and p - bf16(p), both exact in bf16) and a signature of its
    (layer, head) plane; the scores peak at one chosen key (rising with position under the causal mask, or a
    quadratic bump at a chosen frame) and every score is an integer below 2^24, so the fp32 arithmetic is exact;
  * random inputs, held to bounds that follow from the arithmetic of each kernel.
The CPU tests at the top check that the probes are probes.
"""
import math

import pytest
import torch

from whisperlivekit_b200.dims import ModelDimensions

N_CTX = 1500            # encoder frames = cross-attention keys
TILE = 128              # key tile of attn_tc_kernel
LOG2E = 1.4426950408889634
BETA = 32.0             # causal probe: score of key p is BETA * p, so key t - 1 weighs e^-32 against key t
GAMMA = 64.0            # bump probe: score of frame f is -GAMMA * (d(f) - d(f0))^2
CLAMP = 255             # d(f) = clamp(f - center, -CLAMP, CLAMP): keeps every partial sum of the scores below 2^24
NAN = float("nan")

# (dims, alignment heads): a small decoder and large-v3's, two layers each, alignment heads with a head > 0 in layer 1
GEOMS = {
    "small": (ModelDimensions(80, 1500, 384, 6, 1, 51864, 448, 384, 6, 2), [(0, 1), (1, 0), (1, 4)]),
    "large-v3": (ModelDimensions(128, 1500, 1280, 20, 1, 51866, 448, 1280, 20, 2), [(0, 5), (1, 0), (1, 13)]),
}
# ragged batch: a 1-row job (its q tile's padding rows are the next job's), a 40-row job, a 129-row job (a second query
# tile with a single row).  Row positions cover t = 0, 31/32/33 (SIMT lane wrap), 127/128 (key tile) and 447 (last).
RAGGED_ROWS = [1, 40, 129]
RAGGED_OFFSETS = [447, 0, 100]
RAGGED_ALIGN_ROW0 = [447, 3, 300]
# frames of the bump probe: tc key tiles (0, 127/128, 1407/1408), the tail of 1500 = 11 x 128 + 92 (1499), and the
# bounds between the SIMT warps' key ranges (KEYS_PER_WARP = 188: 187/188, 1315/1316); two centers keep |f0 - center|
# within 200 so the clamp never reaches the peak
BUMP_JOBS = [(100, [0, 127, 128, 187, 188]), (1400, [1315, 1316, 1407, 1408, 1499])]
# (backend, type): type 0 = fp32, 1 = bf16
CONFIGS = [("simt", 0), ("simt", 1), ("tcgen05", 1)]
CONFIG_IDS = ["simt-fp32", "simt-bf16", "tcgen05-bf16"]
DTYPE = {0: torch.float32, 1: torch.bfloat16}


# ------------------------------------------------------------------------------------------------------------------
# input builders (fp64 on the CPU)
# ------------------------------------------------------------------------------------------------------------------
def split2(x):
    """Integers below 2^16 -> (hi, lo), both exact in bf16, hi + lo == x."""
    x = torch.as_tensor(x, dtype=torch.float64)
    hi = x.to(torch.bfloat16).double()
    return hi, x - hi


def kslot(layer, head):
    """Group of 8 dims that carries the probe in the K plane of (layer, head): a K read from a neighbouring head or
    from the other layer scores every key 0."""
    return (head + 3 * layer) % 8


def vsig(layer, head):
    """Signature of the V plane of (layer, head) (dim 2 of every row): exact in bf16, distinct for every plane."""
    return float(1 + 32 * layer + head)


def fill_past(kv, n_valid, fill):
    """Cache rows at positions >= n_valid: NaN (the SIMT kernels must never read them) or 'big' = +-1e4 (finite, as
    alloc_session guarantees for the tensor-core kernels, which must give them probability exactly 0)."""
    if fill == "nan":
        kv[..., n_valid:, :] = NAN
    else:
        sign = 1.0 - 2.0 * (torch.arange(kv.shape[-1], dtype=torch.float64) % 2)
        kv[..., n_valid:, :] = 1e4 * sign
    return kv


def causal_cache(L, H, ctx, n_valid, fill):
    """Self-K/V cache [L][2][H][ctx][64]: K of key p = split(p) in the plane's slot (so q = BETA (1, 1) scores it
    BETA * p: the strongest allowed key of the row at position t is t, key t + 1 would win if the mask leaked);
    V of key p = (split(p), signature)."""
    kv = torch.zeros(L, 2, H, ctx, 64, dtype=torch.float64)
    hi, lo = split2(torch.arange(ctx))
    for l in range(L):
        for h in range(H):
            j = 8 * kslot(l, h)
            kv[l, 0, h, :, j], kv[l, 0, h, :, j + 1] = hi, lo
            kv[l, 1, h, :, 0], kv[l, 1, h, :, 1], kv[l, 1, h, :, 2] = hi, lo, vsig(l, h)
    return fill_past(kv, n_valid, fill)


def causal_queries(n_rows, layer, H):
    q = torch.zeros(n_rows, H * 64, dtype=torch.float64)
    for h in range(H):
        q[:, h * 64 + 8 * kslot(layer, h) + torch.arange(2)] = BETA
    return q


def bump_keys(center):
    """[1500, 5]: (hi(d^2), lo(d^2), d, 1, 1), d = clamp(f - center).  With bump_query every product is exact in fp32
    and every partial sum an integer below 2^24 (64 * (255^2 + 2 * 200 * 255 + 200^2) = 1.3e7): the scores are exact
    whatever the order of accumulation."""
    d = (torch.arange(N_CTX, dtype=torch.float64) - center).clamp(-CLAMP, CLAMP)
    hi, lo = split2(d * d)
    one = torch.ones_like(d)
    return torch.stack([hi, lo, d, one, one], dim=1)


def bump_query(f0, center):
    """q . bump_keys(center)[f] = -GAMMA (d(f) - d(f0))^2: a peak at frame f0, its neighbours weigh e^-64."""
    d0 = float(f0 - center)
    assert abs(d0) <= 200
    hi, lo = split2(d0 * d0)
    return GAMMA * torch.tensor([-1.0, -1.0, 2.0 * d0, -hi.item(), -lo.item()], dtype=torch.float64)


def cross_cache(L, H, center):
    """Cross-K/V [L][2][H][1500][64]: the bump keys in the plane's slot, V of frame f = (split(f), signature)."""
    kv = torch.zeros(L, 2, H, N_CTX, 64, dtype=torch.float64)
    keys = bump_keys(center)
    hi, lo = split2(torch.arange(N_CTX))
    for l in range(L):
        for h in range(H):
            j = 8 * kslot(l, h)
            kv[l, 0, h, :, j:j + 5] = keys
            kv[l, 1, h, :, 0], kv[l, 1, h, :, 1], kv[l, 1, h, :, 2] = hi, lo, vsig(l, h)
    return kv


def cross_queries(f0s, center, layer, H):
    q = torch.zeros(len(f0s), H * 64, dtype=torch.float64)
    for t, f0 in enumerate(f0s):
        for h in range(H):
            j = h * 64 + 8 * kslot(layer, h)
            q[t, j:j + 5] = bump_query(f0, center)
    return q


def key_ramp(n):
    """Key-norm multiplier 1, 2, 3, ... per 128-key tile: the maximum of every later tile exceeds the reference maximum
    of the one-pass softmax by more than 2^8 for most rows."""
    return 1.0 + (torch.arange(n) // TILE).double()


# ------------------------------------------------------------------------------------------------------------------
# fp64 references
# ------------------------------------------------------------------------------------------------------------------
def ref_self(q, kvs, layer, n_rows, offsets):
    """Causal softmax(q K^T) V per job over keys 0 .. position (rows beyond the job's last position are not read).
    -> (out [R, H*64], scores per job [H, rows, keys])."""
    outs, scores, r = [], [], 0
    for kv, nr, off in zip(kvs, n_rows, offsets):
        n = off + nr
        K, V = kv[layer, 0, :, :n], kv[layer, 1, :, :n]
        H = K.shape[0]
        qi = q[r:r + nr].reshape(nr, H, 64).transpose(0, 1)
        s = qi @ K.transpose(-1, -2)
        pos = off + torch.arange(nr, device=s.device)
        s = s.masked_fill(torch.arange(n, device=s.device)[None, :] > pos[:, None], -math.inf)
        outs.append((torch.softmax(s, -1) @ V).transpose(0, 1).reshape(nr, H * 64))
        scores.append(s)
        r += nr
    return torch.cat(outs), scores


def ref_cross(q, kvs, layer, n_rows):
    """softmax(q K^T) V over the 1500 frames -> (out [R, H*64], probabilities per job [H, rows, 1500], scores)."""
    outs, probs, scores, r = [], [], [], 0
    for kv, nr in zip(kvs, n_rows):
        K, V = kv[layer, 0], kv[layer, 1]
        H = K.shape[0]
        s = q[r:r + nr].reshape(nr, H, 64).transpose(0, 1) @ K.transpose(-1, -2)
        p = torch.softmax(s, -1)
        outs.append((p @ V).transpose(0, 1).reshape(nr, H * 64))
        probs.append(p)
        scores.append(s)
        r += nr
    return torch.cat(outs), probs, scores


def rescale_rows(s):
    """Rows of fp64 scores [..., keys] (masked keys -inf) on which attn_tc_kernel's one-pass softmax moves its
    reference maximum: a key tile's maximum exceeds the running reference by more than 2^8 (log2 units)."""
    s = s * LOG2E
    m = s[..., :TILE].amax(-1)
    moved = torch.zeros_like(m, dtype=torch.bool)
    for j in range(TILE, s.shape[-1], TILE):
        t = s[..., j:j + TILE].amax(-1)
        need = t > m + 8
        moved |= need
        m = torch.where(need, t, m)
    return moved


def rounded(x, code):
    """What the kernel reads: the fp64 input rounded to the op's type, back in fp64."""
    return x.to(DTYPE[code]).double()


# ------------------------------------------------------------------------------------------------------------------
# CPU: the probes are probes
# ------------------------------------------------------------------------------------------------------------------
def test_position_split_is_exact_in_bf16():
    hi, lo = split2(torch.arange(N_CTX))
    assert torch.equal(rounded(hi, 1), hi) and torch.equal(rounded(lo, 1), lo)
    assert torch.equal(hi + lo, torch.arange(N_CTX, dtype=torch.float64))
    d = bump_keys(100)
    assert torch.equal(rounded(d, 1), d)
    for f0, c in ((0, 100), (1499, 1400), (1316, 1400)):
        assert torch.equal(rounded(bump_query(f0, c), 1), bump_query(f0, c))


@pytest.mark.parametrize("fill", ["nan", "big"])
def test_causal_probe_picks_the_row_position_and_the_mask_matters(fill):
    L, H, ctx = 2, 3, 448
    q = causal_queries(sum(RAGGED_ROWS), 1, H)
    kvs = [causal_cache(L, H, ctx, off + nr, fill) for nr, off in zip(RAGGED_ROWS, RAGGED_OFFSETS)]
    out, scores = ref_self(q, kvs, 1, RAGGED_ROWS, RAGGED_OFFSETS)
    pos = torch.cat([off + torch.arange(nr) for nr, off in zip(RAGGED_ROWS, RAGGED_OFFSETS)]).double()
    for h in range(H):
        assert (out[:, h * 64] + out[:, h * 64 + 1] - pos).abs().max() < 1e-6
        assert torch.all(out[:, h * 64 + 2] == vsig(1, h))
    for s, nr, off in zip(scores, RAGGED_ROWS, RAGGED_OFFSETS):
        assert torch.equal(s.argmax(-1)[0], off + torch.arange(nr))      # the strongest allowed key is the row's own
    # without the mask the next key wins wherever there is one in the cache
    kv = causal_cache(L, H, ctx, 448, fill)
    q0 = causal_queries(1, 1, H)[:, :64]                                  # head 0 of layer 1
    s = q0 @ kv[1, 0, 0].T
    for t in (0, 31, 32, 127, 128, 446):
        assert s[0, : t + 2].argmax().item() == t + 1
    # the K plane of the other layer or of a neighbouring head scores every key alike
    assert torch.all(q0 @ kv[0, 0, 0].T == 0) and torch.all(q0 @ kv[1, 0, 1].T == 0)


def test_bump_probe_peaks_at_the_chosen_frame():
    L, H = 2, 3
    for center, f0s in BUMP_JOBS:
        kv = cross_cache(L, H, center)
        q = cross_queries(f0s, center, 1, H)
        out, probs, scores = ref_cross(q, [kv], 1, [len(f0s)])
        for h in range(H):
            assert torch.equal(probs[0][h].argmax(-1), torch.tensor(f0s))
            assert probs[0][h].amax(-1).min() > 1 - 1e-12
            assert (out[:, h * 64] + out[:, h * 64 + 1] - torch.tensor(f0s)).abs().max() < 1e-20
        # exact integer scores, peak 0, neighbours -64
        s = scores[0][0]
        assert torch.equal(s, s.round()) and s.abs().max() < 2 ** 24
        assert torch.all(s[torch.arange(len(f0s)), torch.tensor(f0s)] == 0)


def test_key_ramp_crosses_the_rescale_threshold():
    """The moving-reference inputs of the GPU tests do take the rescale path on most rows (self and cross)."""
    q, kvs, n_rows, offsets = moving_reference_self_inputs(2, 4, 448)
    _, scores = ref_self(rounded(q, 1), [rounded(k, 1) for k in kvs], 1, n_rows, offsets)
    assert torch.cat([rescale_rows(s).flatten() for s in scores]).double().mean() > 0.5
    q, kvs, n_rows = moving_reference_cross_inputs(2, 4)
    _, _, scores = ref_cross(rounded(q, 1), [rounded(k, 1) for k in kvs], 1, n_rows)
    assert torch.cat([rescale_rows(s).flatten() for s in scores]).double().mean() > 0.5


def moving_reference_self_inputs(L, H, ctx, seed=5):
    """Random q, K, V with key norms growing by one unit per key tile; two jobs of 200 and 100 rows late in the
    context, so every row sees three or four key tiles."""
    g = torch.Generator().manual_seed(seed)
    n_rows, offsets = [200, 100], [248, 340]
    kvs = []
    for nr, off in zip(n_rows, offsets):
        kv = torch.randn(L, 2, H, ctx, 64, generator=g, dtype=torch.float64) * 0.7
        kv[:, 0] *= key_ramp(ctx)[:, None]
        kvs.append(fill_past(kv, off + nr, "big"))
    q = torch.randn(sum(n_rows), H * 64, generator=g, dtype=torch.float64) * 0.7
    return q, kvs, n_rows, offsets


def moving_reference_cross_inputs(L, H, seed=6):
    """Random q, cross-K/V with key norms growing tile by tile over the 1500 frames (one 129-row job: two query
    tiles), like test_encoder_attention_tcgen05_moving_reference."""
    g = torch.Generator().manual_seed(seed)
    kv = torch.randn(L, 2, H, N_CTX, 64, generator=g, dtype=torch.float64) * 0.7
    ramp = torch.ones(N_CTX, dtype=torch.float64)
    ramp[400:] = 1.8; ramp[700:] = 2.6; ramp[1000:] = 3.5; ramp[1300:] = 4.5
    kv[:, 0] *= ramp[:, None]
    q = torch.randn(129, H * 64, generator=g, dtype=torch.float64) * 0.7
    return q, [kv], [129]


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
def bound(backend, code, ref):
    """Elementwise error bound of an output, from the arithmetic of the kernel:
      SIMT fp32  : fp32 math on fp32 inputs, 2e-5 on O(1) outputs (the encoder SIMT test's bound);
      SIMT bf16  : fp32 math on bf16 inputs, only the output is rounded to bf16: 2^-8 |ref| + 1e-4;
      tcgen05    : P is rounded to bf16 before P V (and the output to bf16): 2e-2 on O(1) outputs.
    Measured maxima on a B200 (1000 W) over both geometries and layers, random inputs: self-attention 5.2e-6 / 7.8e-3 /
    1.3e-2, cross-attention 1.2e-6 / 7.8e-3 / 1.2e-2 (SIMT fp32 / SIMT bf16 / tcgen05)."""
    a = ref.abs()
    if backend == "simt":
        return 2e-5 * a.clamp(min=1.0) if code == 0 else a * 2.0 ** -8 + 1e-4
    return 2e-2 * a.clamp(min=1.0)


@pytest.fixture(scope="module", params=list(GEOMS))
def eng(request):
    from whisperlivekit_b200.engine import WhisperEngine
    dims, heads = GEOMS[request.param]
    e = WhisperEngine(dims, None, heads, precision="bf16", max_sessions=1, max_batch=1)
    yield e
    e.close()


def run_op(eng, kind, backend, code, layer, q, kvs, n_rows, offsets, align_row0=None):
    """The op on device copies of the fp64 inputs in the op's type; alignment buffers start as NaN sentinels.
    -> (out fp64, align buffers or None)."""
    dt = DTYPE[code]
    qd = q.to(dt).cuda().contiguous()
    kvd = [kv.to(dt).cuda().contiguous() for kv in kvs]
    out = torch.full_like(qd, NAN)
    aligns = None
    if kind == "cross":
        aligns = [torch.full((len(eng.align_heads), eng.dims.n_text_ctx, N_CTX), NAN, device="cuda") for _ in kvs]
    torch.cuda.synchronize()
    eng.op_decoder_attention(kind, backend, code, layer, qd.data_ptr(), n_rows, offsets, [k.data_ptr() for k in kvd],
                             out.data_ptr(), align_row0, [a.data_ptr() for a in aligns] if aligns else None)
    eng.sync()
    return out.double().cpu(), ([a.cpu() for a in aligns] if aligns else None)


def heads_of(eng, layer):
    """{head: rank} of the engine's alignment heads in `layer`."""
    return {h: r for r, (l, h) in enumerate(eng.align_heads) if l == layer}


def check_align(eng, layer, aligns, probs, n_rows, align_row0, tol=2e-6):
    """Exported rows of this layer's alignment heads = the fp64 softmax; every other row keeps its NaN sentinel."""
    ranks = heads_of(eng, layer)
    worst = 0.0
    for a, p, nr, a0 in zip(aligns, probs, n_rows, align_row0):
        inside = torch.zeros(a.shape[1], dtype=torch.bool)
        inside[a0:a0 + nr] = True
        for rank in range(a.shape[0]):
            head = [h for h, r in ranks.items() if r == rank]
            if not head:
                assert torch.isnan(a[rank]).all(), f"rank {rank} of another layer was written"
                continue
            rows = a[rank, inside].double()
            assert torch.isnan(a[rank, ~inside]).all(), "rows outside [align_row0, align_row0 + n_rows) were written"
            err = (rows - p[head[0]]).abs().max().item()
            worst = max(worst, err)
            assert err < tol, (rank, err)
            assert (rows.sum(-1) - 1).abs().max().item() < 1e-5
    return worst


@pytest.mark.gpu
@pytest.mark.parametrize("backend,code", CONFIGS, ids=CONFIG_IDS)
@pytest.mark.parametrize("case", ["prefill", "step"])
def test_self_attention_causal_probe(eng, backend, code, case):
    """Row t of a job attends to its own key t (never t + 1, never a row past the cache length): the recovered
    position and the V signature of layer 1's planes come out exactly, for every head."""
    D = eng.dims
    L, H, ctx = D.n_text_layer, D.n_text_head, D.n_text_ctx
    n_rows, offsets = (RAGGED_ROWS, RAGGED_OFFSETS) if case == "prefill" else ([1, 1, 1, 1], [0, 32, 128, 447])
    fill = "nan" if backend == "simt" else "big"
    kvs = [causal_cache(L, H, ctx, off + nr, fill) for nr, off in zip(n_rows, offsets)]
    q = causal_queries(sum(n_rows), 1, H)
    out, _ = run_op(eng, "self", backend, code, 1, q, kvs, n_rows, offsets)
    ref, _ = ref_self(rounded(q, code), [rounded(k, code) for k in kvs], 1, n_rows, offsets)
    pos = torch.cat([off + torch.arange(nr) for nr, off in zip(n_rows, offsets)]).double()
    assert not torch.isnan(out).any()
    for h in range(H):
        got = out[:, h * 64] + out[:, h * 64 + 1]
        bad = (got - pos).abs() > 1e-2
        assert not bad.any(), (h, pos[bad][:8].tolist(), got[bad][:8].tolist())
        assert torch.all(out[:, h * 64 + 2] == vsig(1, h)), h
    assert torch.all((out - ref).abs() <= bound(backend, code, ref))


@pytest.mark.gpu
@pytest.mark.parametrize("backend,code", CONFIGS, ids=CONFIG_IDS)
@pytest.mark.parametrize("case", ["prefill", "step"])
def test_cross_attention_bump_probe(eng, backend, code, case):
    """The bump peaks at frames on every tile and warp-range bound: the recovered frame and signature are exact for
    every head, the alignment heads export one-hot rows at align_row0 + t and nothing else."""
    D = eng.dims
    L, H = D.n_text_layer, D.n_text_head
    kvs = [cross_cache(L, H, c) for c, _ in BUMP_JOBS]
    calls = [[f0s for _, f0s in BUMP_JOBS]] if case == "prefill" else \
        [[[a], [b]] for a, b in zip(BUMP_JOBS[0][1], BUMP_JOBS[1][1])]
    for layer in (1, 0):
        for f0s in calls:
            n_rows = [len(f) for f in f0s]
            align_row0 = [5, D.n_text_ctx - n_rows[1]]
            q = torch.cat([cross_queries(f, c, layer, H) for f, (c, _) in zip(f0s, BUMP_JOBS)])
            out, aligns = run_op(eng, "cross", backend, code, layer, q, kvs, n_rows, [0, 0], align_row0)
            ref, probs, _ = ref_cross(rounded(q, code), [rounded(k, code) for k in kvs], layer, n_rows)
            want = torch.tensor(sum(f0s, []), dtype=torch.float64)
            for h in range(H):
                got = out[:, h * 64] + out[:, h * 64 + 1]
                assert (got - want).abs().max() < 1e-2, (layer, h, want.tolist(), got.tolist())
                assert torch.all(out[:, h * 64 + 2] == vsig(layer, h)), (layer, h)
            assert torch.all((out - ref).abs() <= bound(backend, code, ref))
            check_align(eng, layer, aligns, probs, n_rows, align_row0)
            for a, f, a0 in zip(aligns, f0s, align_row0):
                for rank in heads_of(eng, layer).values():
                    assert torch.equal(a[rank, a0:a0 + len(f)].argmax(-1), torch.tensor(f))


def random_self_inputs(L, H, ctx, code, backend, seed):
    g = torch.Generator().manual_seed(seed)
    kvs = [fill_past(torch.randn(L, 2, H, ctx, 64, generator=g, dtype=torch.float64) * 0.8, off + nr,
                     "nan" if backend == "simt" else "big")
           for nr, off in zip(RAGGED_ROWS, RAGGED_OFFSETS)]
    q = torch.randn(sum(RAGGED_ROWS), H * 64, generator=g, dtype=torch.float64) * 0.8
    return q, kvs


@pytest.mark.gpu
@pytest.mark.parametrize("backend,code", CONFIGS, ids=CONFIG_IDS)
def test_self_attention_random(eng, backend, code):
    """Random q / K / V (std 0.8) over the ragged batch, both layers, against the fp64 causal softmax (bounds and
    measured maxima: bound())."""
    D = eng.dims
    q, kvs = random_self_inputs(D.n_text_layer, D.n_text_head, D.n_text_ctx, code, backend, seed=code + 7)
    for layer in range(D.n_text_layer):
        out, _ = run_op(eng, "self", backend, code, layer, q, kvs, RAGGED_ROWS, RAGGED_OFFSETS)
        ref, _ = ref_self(rounded(q, code), [rounded(k, code) for k in kvs], layer, RAGGED_ROWS, RAGGED_OFFSETS)
        err = (out - ref).abs()
        print(f"self {backend}-{code} d={D.n_text_state} layer {layer}: max err {err.max().item():.3e}")
        assert torch.all(err <= bound(backend, code, ref)), err.max().item()


@pytest.mark.gpu
@pytest.mark.parametrize("backend,code", CONFIGS, ids=CONFIG_IDS)
def test_cross_attention_random(eng, backend, code):
    """Random q / K (std 0.5) and V (std 1) over the ragged batch, both layers: outputs against the fp64 softmax,
    alignment rows within 2e-6 of it (fp32 scores of 64 exact products, expf, one division) and summing to 1 within
    1e-5; on the tcgen05 backend the alignment rows are bit-identical to the SIMT backend's (the same kernel makes
    them).  Measured on a B200 (1000 W): alignment rows within 3.6e-7 of fp64; outputs in bound()'s docstring."""
    D = eng.dims
    L, H = D.n_text_layer, D.n_text_head
    g = torch.Generator().manual_seed(11 + code)
    kvs = []
    for _ in RAGGED_ROWS:
        kv = torch.randn(L, 2, H, N_CTX, 64, generator=g, dtype=torch.float64)
        kv[:, 0] *= 0.5
        kvs.append(kv)
    q = torch.randn(sum(RAGGED_ROWS), H * 64, generator=g, dtype=torch.float64) * 0.5
    for layer in range(L):
        out, aligns = run_op(eng, "cross", backend, code, layer, q, kvs, RAGGED_ROWS, RAGGED_OFFSETS, RAGGED_ALIGN_ROW0)
        ref, probs, _ = ref_cross(rounded(q, code), [rounded(k, code) for k in kvs], layer, RAGGED_ROWS)
        err = (out - ref).abs()
        lim = bound(backend, code, ref)
        if backend == "tcgen05":                    # alignment heads run on the SIMT kernel
            for h in heads_of(eng, layer):
                lim[:, h * 64:(h + 1) * 64] = bound("simt", code, ref[:, h * 64:(h + 1) * 64])
        worst = check_align(eng, layer, aligns, probs, RAGGED_ROWS, RAGGED_ALIGN_ROW0)
        print(f"cross {backend}-{code} d={D.n_text_state} layer {layer}: max err {err.max().item():.3e}, "
              f"align rows {worst:.3e}")
        assert torch.all(err <= lim), err.max().item()
        if backend == "tcgen05":
            _, simt = run_op(eng, "cross", "simt", code, layer, q, kvs, RAGGED_ROWS, RAGGED_OFFSETS, RAGGED_ALIGN_ROW0)
            for a, b in zip(aligns, simt):
                assert torch.equal(a.view(torch.int32), b.view(torch.int32))


@pytest.mark.gpu
def test_self_attention_tcgen05_moving_reference(eng):
    """MODE_SELF with key norms growing tile by tile: most rows move their softmax reference (asserted from the fp64
    scores), the result stays within the tcgen05 bound (measured on a B200 at 1000 W: 1.3e-2)."""
    D = eng.dims
    q, kvs, n_rows, offsets = moving_reference_self_inputs(D.n_text_layer, D.n_text_head, D.n_text_ctx)
    out, _ = run_op(eng, "self", "tcgen05", 1, 1, q, kvs, n_rows, offsets)
    ref, scores = ref_self(rounded(q, 1), [rounded(k, 1) for k in kvs], 1, n_rows, offsets)
    assert torch.cat([rescale_rows(s).flatten() for s in scores]).double().mean() > 0.5
    err = (out - ref).abs()
    print(f"self moving reference d={D.n_text_state}: max err {err.max().item():.3e}")
    assert torch.all(err <= bound("tcgen05", 1, ref)), err.max().item()


@pytest.mark.gpu
def test_cross_attention_tcgen05_moving_reference(eng):
    """MODE_CROSS with key norms growing tile by tile over the 1500 frames: most rows move their softmax reference
    (measured on a B200 at 1000 W: 1.4e-2 against the 2e-2 bound)."""
    D = eng.dims
    q, kvs, n_rows = moving_reference_cross_inputs(D.n_text_layer, D.n_text_head)
    out, aligns = run_op(eng, "cross", "tcgen05", 1, 1, q, kvs, n_rows, [0], [0])
    ref, probs, scores = ref_cross(rounded(q, 1), [rounded(k, 1) for k in kvs], 1, n_rows)
    tc_heads = [h for h in range(D.n_text_head) if h not in heads_of(eng, 1)]
    assert rescale_rows(scores[0][tc_heads]).double().mean() > 0.5
    cols = torch.cat([torch.arange(h * 64, (h + 1) * 64) for h in tc_heads])
    err = (out[:, cols] - ref[:, cols]).abs()
    print(f"cross moving reference d={D.n_text_state}: max err {err.max().item():.3e}")
    assert torch.all(err <= bound("tcgen05", 1, ref[:, cols])), err.max().item()
    check_align(eng, 1, aligns, probs, n_rows, [0])


@pytest.mark.gpu
def test_decoder_attention_rejects_bad_input(eng):
    """Bad arguments come back as an error status with a message, never as a launch."""
    from whisperlivekit_b200._lib import WlkError, check
    D = eng.dims
    ctx, L, H = D.n_text_ctx, D.n_text_layer, D.n_text_head
    q = torch.zeros(4, H * 64, device="cuda", dtype=torch.bfloat16)
    out = torch.zeros_like(q)
    skv = torch.zeros(L, 2, H, ctx, 64, device="cuda", dtype=torch.bfloat16)
    xkv = torch.zeros(L, 2, H, N_CTX, 64, device="cuda", dtype=torch.bfloat16)
    al = torch.zeros(len(eng.align_heads), ctx, N_CTX, device="cuda")

    def call(kind="self", backend="simt", code=1, layer=0, qp=None, n_rows=(4,), offsets=(0,), kv=None, outp=None,
             align_row0=(0,), align=None):
        kvp = kv if kv is not None else (skv if kind == "self" else xkv).data_ptr()
        eng.op_decoder_attention(kind, backend, code, layer, q.data_ptr() if qp is None else qp, list(n_rows),
                                 list(offsets), [kvp], out.data_ptr() if outp is None else outp, list(align_row0),
                                 [al.data_ptr() if align is None else align])

    call()
    call(kind="cross", backend="tcgen05")
    eng.sync()
    bad = [dict(offsets=(ctx - 3,)), dict(offsets=(-1,)), dict(n_rows=(0,)),
           dict(kind="cross", align_row0=(ctx - 3,)), dict(layer=L), dict(layer=-1), dict(backend="tcgen05", code=0),
           dict(code=2), dict(qp=q.data_ptr() + 2), dict(outp=out.data_ptr() + 8), dict(kv=skv.data_ptr() + 4),
           dict(kind="cross", align=al.data_ptr() + 4), dict(kv=0), dict(qp=0), dict(kind="cross", align=0)]
    for kw in bad:
        with pytest.raises(WlkError):
            call(**kw)
    for kind, backend, what in ((2, 1, "kind"), (0, 3, "backend")):
        with pytest.raises(WlkError, match=what):
            check(eng.lib.wlk_op_decoder_attention(eng.h, kind, backend, 1, 0, q.data_ptr(), 1, None, None, None, None,
                                                   None, out.data_ptr()))
    eng.sync()
