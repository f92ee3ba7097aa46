"""GPU: op-level checks of the hand-written kernels through the C ABI (wlk_op_*),
against plain torch fp32 references of the same op."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from whisperlivekit_b200.dims import DIMS


@pytest.fixture(scope="module")
def eng():
    from whisperlivekit_b200.engine import WhisperEngine
    e = WhisperEngine(DIMS["micro"], None, [(0, 0)], precision="bf16", max_sessions=1, max_batch=1)
    yield e
    e.close()


def _gemm(eng, backend, A, W, bias, gelu, out_dtype):
    M, K = A.shape
    N = W.shape[0]
    Cm = torch.empty(M, N, device="cuda", dtype=out_dtype)
    code = {torch.float32: 0, torch.bfloat16: 1}
    torch.cuda.synchronize()
    eng.op_gemm(backend, A.data_ptr(), code[A.dtype], A.stride(0), W.data_ptr(), code[W.dtype], W.stride(0),
                bias.data_ptr() if bias is not None else None, Cm.data_ptr(), code[out_dtype], Cm.stride(0),
                M, N, K, gelu)
    eng.sync()
    return Cm


def _ref(A, W, bias, gelu):
    r = A.float() @ W.float().t()
    if bias is not None:
        r = r + bias
    if gelu:
        r = torch.nn.functional.gelu(r)
    return r


@pytest.mark.parametrize("M,N,K", [(128, 128, 64), (1500, 384, 384), (37, 51, 20), (16, 1280, 1280), (3, 51864, 128)])
@pytest.mark.parametrize("gelu", [False, True])
def test_gemm_simt_fp32(eng, M, N, K, gelu):
    g = torch.Generator(device="cuda").manual_seed(M * 7 + N)
    A = torch.randn(M, K, device="cuda", generator=g)
    W = torch.randn(N, K, device="cuda", generator=g) / K ** 0.5
    b = torch.randn(N, device="cuda", generator=g)
    out = _gemm(eng, "simt", A, W, b, gelu, torch.float32)
    ref = _ref(A.double(), W.double(), b.double(), gelu).float() if not gelu else _ref(A, W, b, gelu)
    assert (out - ref).abs().max().item() < 2e-4 * max(1.0, ref.abs().max().item())


SHAPES_TC = [(128, 256, 64), (256, 256, 128), (1500, 1280, 1280), (3000, 384, 240), (1000, 3840, 1280),
             (129, 264, 72), (64, 128, 5120), (4500, 5120, 1280), (12000, 1280, 5120),
             (16, 3840, 1280), (64, 1280, 1280), (1, 51864, 384), (200, 1280, 5120)]


@pytest.mark.parametrize("M,N,K", SHAPES_TC)
def test_gemm_tcgen05_bf16(eng, M, N, K):
    """tcgen05 GEMM vs fp32 reference on the same bf16-rounded operands: only the fp32
    accumulation order differs, so the bound is tight (1e-3 relative to the output scale)."""
    g = torch.Generator(device="cuda").manual_seed(M + N + K)
    A = torch.randn(M, K, device="cuda", generator=g).bfloat16()
    W = (torch.randn(N, K, device="cuda", generator=g) / K ** 0.5).bfloat16()
    b = torch.randn(N, device="cuda", generator=g)
    for gelu in (False, True):
        out = _gemm(eng, "tcgen05", A, W, b, gelu, torch.float32)
        ref = _ref(A, W, b, gelu)
        err = (out - ref).abs().max().item()
        assert err < 1e-3 * max(1.0, ref.abs().max().item()), (M, N, K, gelu, err)
    out_bf = _gemm(eng, "tcgen05", A, W, b, False, torch.bfloat16)
    ref = _ref(A, W, b, False)
    assert (out_bf.float() - ref).abs().max().item() < 2e-2 * max(1.0, ref.abs().max().item())
    simt = _gemm(eng, "simt", A, W, b, False, torch.float32)
    assert (simt - _gemm(eng, "tcgen05", A, W, b, False, torch.float32)).abs().max().item() < 1e-3 * max(1.0, ref.abs().max().item())


def test_gemm_tcgen05_strided_overlapping_rows(eng):
    """The conv stem feeds the GEMM overlapping rows (pitch < row length) through the TMA map."""
    g = torch.Generator(device="cuda").manual_seed(5)
    base = torch.randn(3002 * 80, device="cuda", generator=g).bfloat16()
    A = torch.as_strided(base, (3000, 240), (80, 1))
    W = (torch.randn(384, 240, device="cuda", generator=g) / 15).bfloat16()
    out = _gemm(eng, "tcgen05", A, W, None, False, torch.float32)
    ref = A.float() @ W.float().t()
    assert (out - ref).abs().max().item() < 1e-3 * ref.abs().max().item()


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_encoder_attention_simt(eng, dtype):
    d, H, B = 128, 2, 2
    g = torch.Generator(device="cuda").manual_seed(3)
    qkv = (torch.randn(B * 1500, 3 * d, device="cuda", generator=g) * 0.8).to(dtype)
    out = torch.empty(B * 1500, d, device="cuda", dtype=dtype)
    torch.cuda.synchronize()
    eng.op_encoder_attention("simt", qkv.data_ptr(), 0 if dtype == torch.float32 else 1, B, out.data_ptr())
    eng.sync()
    x = qkv.float().view(B, 1500, 3, H, 64)
    q, k, v = x[:, :, 0].transpose(1, 2), x[:, :, 1].transpose(1, 2), x[:, :, 2].transpose(1, 2)
    ref = (torch.softmax(q @ k.transpose(-1, -2), dim=-1) @ v).transpose(1, 2).reshape(B * 1500, d)
    tol = 2e-5 if dtype == torch.float32 else 1e-2
    assert (out.float() - ref).abs().max().item() < tol


@pytest.mark.parametrize("d,H,B", [(128, 2, 1), (384, 6, 2), (1280, 20, 1)])
def test_encoder_attention_tcgen05(eng, d, H, B):
    """Fused tcgen05 attention vs fp32 softmax(QK^T)V on the same bf16 inputs.  P is rounded to
    bf16 before the PV product (8 mantissa bits): tolerance 2e-2 on outputs of O(1)."""
    from whisperlivekit_b200.dims import ModelDimensions
    from whisperlivekit_b200.engine import WhisperEngine
    e2 = WhisperEngine(ModelDimensions(80, 1500, d, H, 1, 51864, 448, 64, 1, 1), None, [(0, 0)], precision="bf16",
                       max_sessions=1, max_batch=1)
    g = torch.Generator(device="cuda").manual_seed(d)
    qkv = (torch.randn(B * 1500, 3 * d, device="cuda", generator=g) * 0.8).bfloat16()
    out = torch.full((B * 1500, d), float("nan"), device="cuda", dtype=torch.bfloat16)
    torch.cuda.synchronize()
    e2.op_encoder_attention("tcgen05", qkv.data_ptr(), 1, B, out.data_ptr())
    e2.sync()
    x = qkv.float().view(B, 1500, 3, H, 64)
    q, k, v = x[:, :, 0].transpose(1, 2), x[:, :, 1].transpose(1, 2), x[:, :, 2].transpose(1, 2)
    ref = (torch.softmax(q @ k.transpose(-1, -2), dim=-1) @ v).transpose(1, 2).reshape(B * 1500, d)
    assert not torch.isnan(out.float()).any()
    assert (out.float() - ref).abs().max().item() < 2e-2
    e2.close()


def test_encoder_attention_tcgen05_moving_reference():
    """The one-pass softmax keeps a reference maximum per row and only moves it (rescaling O and l in TMEM and redoing the
    tile) when a key tile exceeds it by more than 2^8.  Random inputs almost never take that path: here the keys of later
    tiles are scaled up so that most rows move their reference several times, at different tiles."""
    from whisperlivekit_b200.dims import ModelDimensions
    from whisperlivekit_b200.engine import WhisperEngine
    d, H, B = 256, 4, 2
    e2 = WhisperEngine(ModelDimensions(80, 1500, d, H, 1, 51864, 448, 64, 1, 1), None, [(0, 0)], precision="bf16",
                       max_sessions=1, max_batch=1)
    g = torch.Generator(device="cuda").manual_seed(77)
    x = torch.randn(B, 1500, 3, H, 64, device="cuda", generator=g) * 0.7
    ramp = torch.ones(1500, device="cuda")
    ramp[400:] = 1.8; ramp[700:] = 2.6; ramp[1000:] = 3.5; ramp[1300:] = 4.5       # key norms grow tile by tile
    x[:, :, 1] *= ramp[None, :, None, None]
    x[1, :, 1, 1] *= torch.linspace(1.0, 0.2, 1500, device="cuda")[:, None]         # ... and one head where they shrink
    qkv = x.reshape(B * 1500, 3 * d).bfloat16()
    out = torch.full((B * 1500, d), float("nan"), device="cuda", dtype=torch.bfloat16)
    torch.cuda.synchronize()
    e2.op_encoder_attention("tcgen05", qkv.data_ptr(), 1, B, out.data_ptr())
    e2.sync()
    xf = qkv.float().view(B, 1500, 3, H, 64)
    q, k, v = xf[:, :, 0].transpose(1, 2), xf[:, :, 1].transpose(1, 2), xf[:, :, 2].transpose(1, 2)
    s = q @ k.transpose(-1, -2)
    jump = (s[..., 1280:].amax(-1) - s[..., :128].amax(-1)) * 1.4427                # log2 units, last tile vs first
    assert (jump > 8).float().mean().item() > 0.5                                   # the path under test is really taken
    ref = (torch.softmax(s, dim=-1) @ v).transpose(1, 2).reshape(B * 1500, d)
    assert not torch.isnan(out.float()).any()
    assert (out.float() - ref).abs().max().item() < 3e-2
    e2.close()


@pytest.mark.parametrize("M,N,K", [(256, 256, 64), (512, 512, 256), (1500, 1280, 1280), (3000, 384, 240),
                                   (257, 300, 72), (24000, 1280, 1280), (4500, 5120, 1280)])
def test_gemm_tcgen05_cta_pair(eng, M, N, K):
    """cta_group::2 kernel (256x256 tiles over 2-CTA clusters) vs fp32 reference and vs the 1-CTA kernel."""
    g = torch.Generator(device="cuda").manual_seed(M + 3 * N + K)
    A = torch.randn(M, K, device="cuda", generator=g).bfloat16()
    W = (torch.randn(N, K, device="cuda", generator=g) / K ** 0.5).bfloat16()
    b = torch.randn(N, device="cuda", generator=g)
    out = _gemm(eng, "tcgen05_pair", A, W, b, True, torch.float32)
    ref = _ref(A, W, b, True)
    assert not torch.isnan(out).any()
    assert (out - ref).abs().max().item() < 1e-3 * max(1.0, ref.abs().max().item())
    one = _gemm(eng, "tcgen05_1cta", A, W, b, True, torch.float32)
    assert (out - one).abs().max().item() < 1e-4 * max(1.0, ref.abs().max().item())


@pytest.mark.parametrize("M,N,K", [(16, 1280, 1280), (64, 1280, 5120), (1, 384, 1536), (48, 512, 512)])
def test_gemm_tcgen05_split_k_in_place(eng, M, N, K):
    """Decoder-shaped GEMMs updating the fp32 residual stream in place (x += A W^T + b): the short/narrow
    case is split along K with fp32 atomics."""
    g = torch.Generator(device="cuda").manual_seed(M + N + K)
    A = torch.randn(M, K, device="cuda", generator=g).bfloat16()
    W = (torch.randn(N, K, device="cuda", generator=g) / K ** 0.5).bfloat16()
    b = torch.randn(N, device="cuda", generator=g)
    x0 = torch.randn(M, N, device="cuda", generator=g)
    x = x0.clone()
    torch.cuda.synchronize()
    eng.op_gemm("tcgen05", A.data_ptr(), 1, K, W.data_ptr(), 1, K, b.data_ptr(), x.data_ptr(), 0, N, M, N, K, 2)
    eng.sync()
    ref = x0 + A.float() @ W.float().t() + b
    assert (x - ref).abs().max().item() < 1e-3 * max(1.0, ref.abs().max().item())


# ---- one-query-tile encoder attention and the split-operand (bf16x3) kernels, against fp64 -----------------------------
def _enc_engine(d, H):
    from whisperlivekit_b200.dims import ModelDimensions
    from whisperlivekit_b200.engine import WhisperEngine
    return WhisperEngine(ModelDimensions(80, 1500, d, H, 1, 51864, 448, 64, 1, 1), None, [(0, 0)], precision="bf16",
                         max_sessions=1, max_batch=1)


def _enc_ref64(qkv, B, H):
    """fp64 softmax(Q K^T) V of the fused [B*1500, 3d] buffer -> (out [B*1500, d], scores [B, H, 1500, 1500])."""
    x = qkv.double().view(B, 1500, 3, H, 64)
    q, k, v = x[:, :, 0].transpose(1, 2), x[:, :, 1].transpose(1, 2), x[:, :, 2].transpose(1, 2)
    s = q @ k.transpose(-1, -2)
    return (torch.softmax(s, dim=-1) @ v).transpose(1, 2).reshape(B * 1500, H * 64), s


def _enc_run(e, backend, qkv, code, B, d):
    out = torch.full((B * 1500, d), float("nan"), device="cuda", dtype=torch.float32 if code != 1 else torch.bfloat16)
    torch.cuda.synchronize()
    e.op_encoder_attention(backend, qkv.data_ptr(), code, B, out.data_ptr())
    e.sync()
    return out.double()


def _enc_inputs(B, H, seed, ramp):
    """fp32 q|k|v [B*1500, 3d] of std 0.7-0.8; ramp: key norms grow tile by tile (and shrink on one head), as in
    test_encoder_attention_tcgen05_moving_reference, so that most rows move their softmax reference."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    if not ramp:
        return torch.randn(B * 1500, 3 * H * 64, device="cuda", generator=g) * 0.8
    x = torch.randn(B, 1500, 3, H, 64, device="cuda", generator=g) * 0.7
    r = torch.ones(1500, device="cuda")
    r[400:] = 1.8; r[700:] = 2.6; r[1000:] = 3.5; r[1300:] = 4.5
    x[:, :, 1] *= r[None, :, None, None]
    x[1 % B, :, 1, 1] *= torch.linspace(1.0, 0.2, 1500, device="cuda")[:, None]
    return x.reshape(B * 1500, 3 * H * 64)


def _moving_share(s):
    jump = (s[..., 1280:].amax(-1) - s[..., :128].amax(-1)) * 1.4427                # log2 units, last tile vs first
    return (jump > 8).double().mean().item()


@pytest.mark.parametrize("d,H,B", [(128, 2, 1), (384, 6, 2), (1280, 20, 1)])
def test_encoder_attention_tcgen05_one_tile(d, H, B):
    """The one-query-tile kernel (backend 3: the kernel body of the decoder prefills and of the bf16x3 mode; the
    encoder's default is the two-tile kernel) vs fp64 on the same bf16 inputs: 2e-2 on O(1) outputs (P in bf16).
    Measured on a B200 (1000 W): 1.3e-2 to 1.4e-2."""
    e2 = _enc_engine(d, H)
    qkv = _enc_inputs(B, H, d + 1, ramp=False).bfloat16()
    out = _enc_run(e2, "tcgen05_1tile", qkv, 1, B, d)
    ref, _ = _enc_ref64(qkv, B, H)
    assert not torch.isnan(out).any()
    err = (out - ref).abs().max().item()
    print(f"one-tile encoder attention d={d} B={B}: max err {err:.3e}")
    assert err < 2e-2
    e2.close()


def test_encoder_attention_tcgen05_one_tile_moving_reference():
    """The one-tile kernel on inputs where most rows move their softmax reference (rescale of O and l in TMEM).
    Measured on a B200 (1000 W): 1.4e-2."""
    d, H, B = 256, 4, 2
    e2 = _enc_engine(d, H)
    qkv = _enc_inputs(B, H, 77, ramp=True).bfloat16()
    out = _enc_run(e2, "tcgen05_1tile", qkv, 1, B, d)
    ref, s = _enc_ref64(qkv, B, H)
    assert _moving_share(s) > 0.5                                                    # the path under test is taken
    assert not torch.isnan(out).any()
    err = (out - ref).abs().max().item()
    print(f"one-tile encoder attention, moving reference: max err {err:.3e}")
    assert err < 2e-2
    e2.close()


@pytest.mark.parametrize("ramp", [False, True], ids=["random", "moving_reference"])
def test_encoder_attention_bf16x3(ramp):
    """Split-plane attention (type 2: bf16 hi plane with the lo plane behind it, fp32 out) vs fp64 on the raw fp32
    inputs: within 1e-3, and at most 1/10 of the one-tile bf16 kernel's error on the same inputs -- Q K^T and P V
    each take three MMAs (hi hi + lo hi + hi lo), so every dropped lo term shows.  Measured on a B200 (1000 W):
    1.0e-4 (random) and 2.8e-4 (ramp) against 5.3e-2 and 1.4e-1 for the bf16 kernel."""
    d, H, B = 384, 6, 2
    e2 = _enc_engine(d, H)
    x = _enc_inputs(B, H, 91, ramp)
    hi = x.bfloat16()
    planes = torch.cat([hi, (x - hi.float()).bfloat16()])
    ref, s = _enc_ref64(x, B, H)
    if ramp:
        assert _moving_share(s) > 0.5
    out = _enc_run(e2, "tcgen05", planes, 2, B, d)
    err = (out - ref).abs().max().item()
    err_bf16 = (_enc_run(e2, "tcgen05_1tile", hi, 1, B, d) - ref).abs().max().item()
    print(f"bf16x3 encoder attention ({'ramp' if ramp else 'random'}): max err {err:.3e}, bf16 one-tile {err_bf16:.3e}")
    assert not torch.isnan(out).any()
    assert err < 1e-3 and err < err_bf16 / 10, (err, err_bf16)
    e2.close()


def _x3_check(eng, backend, A, A_bf, W, b, in_place=False):
    """bf16x3 GEMM (w_type 2: W's hi plane, the lo plane right behind it; fp32 A split on the fly) vs fp64 on the fp32
    operands: |err| <= 2e-4 max(1, |ref|) elementwise (~16 mantissa bits per product), and at most 1/20 of the plain
    bf16 kernel's error on the same operands, which only holds when both lo-plane MMAs contribute.  Measured on a B200
    (1000 W): at most 3.5e-5, against 9e-3 to 1.3e-2 for the bf16 kernel."""
    M, K = A.shape
    N = W.shape[0]
    g = torch.Generator(device="cuda").manual_seed(M + N)
    x0 = torch.randn(M, N, device="cuda", generator=g) if in_place else torch.zeros(M, N, device="cuda")
    ref = x0.double() + A.double() @ W.double().t() + b.double()
    W_hi = W.bfloat16()
    planes = torch.cat([W_hi, (W - W_hi.float()).bfloat16()])
    flags = 2 if in_place else 0
    out3, outb = x0.clone(), x0.clone()
    torch.cuda.synchronize()
    eng.op_gemm(backend, A.data_ptr(), 0, A.stride(0), planes.data_ptr(), 2, K, b.data_ptr(), out3.data_ptr(), 0, N,
                M, N, K, flags)
    eng.op_gemm(backend, A_bf.data_ptr(), 1, A_bf.stride(0), W_hi.data_ptr(), 1, K, b.data_ptr(), outb.data_ptr(), 0, N,
                M, N, K, flags)
    eng.sync()
    err3 = (out3.double() - ref).abs()
    errb = (outb.double() - ref).abs().max().item()
    print(f"bf16x3 gemm {backend} {M}x{N}x{K}{' in place' if in_place else ''}: max err {err3.max().item():.3e}, "
          f"bf16 {errb:.3e}")
    assert torch.all(err3 <= 2e-4 * ref.abs().clamp(min=1.0)), err3.max().item()
    assert err3.max().item() <= errb / 20, (err3.max().item(), errb)


X3_SHAPES = [("tcgen05", 16, 1280, 5120), ("tcgen05", 129, 264, 72), ("tcgen05", 1500, 1280, 1280),
             ("tcgen05", 3000, 5120, 1280), ("tcgen05_1cta", 1500, 1280, 1280), ("tcgen05_1cta", 129, 264, 72),
             ("tcgen05_1cta", 64, 1280, 5120), ("tcgen05_pair", 512, 512, 256), ("tcgen05_pair", 257, 300, 72),
             ("tcgen05_pair", 1000, 3840, 1280)]


@pytest.mark.parametrize("backend,M,N,K", X3_SHAPES)
def test_gemm_bf16x3(eng, backend, M, N, K):
    """Auto tiles (split-K for 16 x 1280 x 5120, the CTA pair for 3000 x 5120), the one-CTA and the CTA-pair kernel."""
    g = torch.Generator(device="cuda").manual_seed(M * 3 + N + K)
    A = torch.randn(M, K, device="cuda", generator=g)
    W = torch.randn(N, K, device="cuda", generator=g) / K ** 0.5
    b = torch.randn(N, device="cuda", generator=g)
    _x3_check(eng, backend, A, A.bfloat16(), W, b)


@pytest.mark.parametrize("M,N,K", [(16, 1280, 1280), (64, 1280, 5120), (48, 512, 512)])
def test_gemm_bf16x3_in_place(eng, M, N, K):
    """x += A W^T + b on the fp32 residual stream, as the bf16x3 decoder runs it (split-K with fp32 atomics for K 5120)."""
    g = torch.Generator(device="cuda").manual_seed(M + N + K + 1)
    A = torch.randn(M, K, device="cuda", generator=g)
    W = torch.randn(N, K, device="cuda", generator=g) / K ** 0.5
    b = torch.randn(N, device="cuda", generator=g)
    _x3_check(eng, "tcgen05", A, A.bfloat16(), W, b, in_place=True)


def test_gemm_bf16x3_strided_overlapping_rows(eng):
    """The conv stem's view with overlapping rows (lda 80 < K 240): the split covers the whole underlying range."""
    g = torch.Generator(device="cuda").manual_seed(6)
    base = torch.randn(3002 * 80, device="cuda", generator=g)
    A = torch.as_strided(base, (3000, 240), (80, 1))
    A_bf = torch.as_strided(base.bfloat16(), (3000, 240), (80, 1))
    W = torch.randn(384, 240, device="cuda", generator=g) / 15
    b = torch.randn(384, device="cuda", generator=g)
    _x3_check(eng, "tcgen05", A, A_bf, W, b)
