"""-m gpu: every ViT operator of libdss_b200 against a plain PyTorch fp32 reference of the same op
(and the tcgen05 GEMM against the in-GPU CUDA-core checker on identical fp16 operands)."""
import math

import pytest
import torch

from conftest import load_pkg

pytestmark = pytest.mark.gpu


def _gemm(lib, _lib, fn, A, Wt, bias, out, epi, aux=None, rin=0, rout=0):
    M, K = A.shape
    N = Wt.shape[0]
    _lib.check(fn(A.data_ptr(), Wt.data_ptr(), bias.data_ptr(), out.data_ptr(), M, N, K, epi,
                  None if aux is None else aux.data_ptr(), rin, rout, _lib.stream_ptr()), "gemm")
    torch.cuda.synchronize()


@pytest.mark.parametrize("M,N,K", [(128, 128, 64), (256, 384, 384), (901, 1152, 384), (1802, 1536, 384),
                                   (901, 384, 1536), (197, 384, 768), (3 * 901, 384, 384), (77, 96, 192)])
def test_gemm_bias_f32_vs_torch_and_simt(cuda, M, N, K):
    _lib = load_pkg("_lib"); lib = _lib.load()
    g = torch.Generator(device="cuda").manual_seed(M * 7 + N)
    A = torch.randn(M, K, device=cuda, generator=g).half()
    Wt = (torch.randn(N, K, device=cuda, generator=g) * 0.05).half()
    bias = torch.randn(N, device=cuda, generator=g)
    out = torch.full((M, N), float("nan"), device=cuda)
    ref = torch.full((M, N), float("nan"), device=cuda)
    _gemm(lib, _lib, lib.dss_op_gemm_f16, A, Wt, bias, out, _lib.EPI_BIAS_F32)
    _gemm(lib, _lib, lib.dss_op_gemm_f16_simt, A, Wt, bias, ref, _lib.EPI_BIAS_F32)
    tref = A.float() @ Wt.float().T + bias
    assert torch.isfinite(out).all(), f"non-finite outputs: {(~torch.isfinite(out)).sum().item()} of {out.numel()}"
    err_simt = (out - ref).abs().max().item()
    err_torch = (out - tref).abs().max().item()
    scale = tref.abs().max().item()
    print(f"gemm {M}x{N}x{K}: |tc-simt|={err_simt:.3e} |tc-torch|={err_torch:.3e} scale={scale:.3f}")
    assert err_simt <= 2e-4 * max(1.0, scale), (err_simt, scale)   # same fp16 operands, fp32 accumulate (order differs)
    assert err_torch <= 2e-4 * max(1.0, scale)


def test_gemm_epilogues(cuda):
    _lib = load_pkg("_lib"); lib = _lib.load()
    g = torch.Generator(device="cuda").manual_seed(5)
    B, T, d = 3, 197, 384
    M = B * T
    A = torch.randn(M, d, device=cuda, generator=g).half()
    Wt = (torch.randn(d, d, device=cuda, generator=g) * 0.05).half()
    bias = torch.randn(d, device=cuda, generator=g)
    acc = A.float() @ Wt.float().T + bias
    # f16 out
    o16 = torch.zeros(M, d, device=cuda, dtype=torch.float16)
    _gemm(lib, _lib, lib.dss_op_gemm_f16, A, Wt, bias, o16, _lib.EPI_BIAS_F16)
    assert (o16.float() - acc).abs().max().item() <= 2e-3 * acc.abs().max().item()
    # gelu f16
    _gemm(lib, _lib, lib.dss_op_gemm_f16, A, Wt, bias, o16, _lib.EPI_BIAS_GELU_F16)
    ge = torch.nn.functional.gelu(acc)
    assert (o16.float() - ge).abs().max().item() <= 2e-3 * ge.abs().max().item()
    # residual f32 in place
    x = torch.randn(M, d, device=cuda, generator=g)
    x0 = x.clone()
    _gemm(lib, _lib, lib.dss_op_gemm_f16, A, Wt, bias, x, _lib.EPI_BIAS_RESID_F32)
    assert (x - (x0 + acc)).abs().max().item() <= 2e-4 * acc.abs().max().item()
    # drop-cls remap: rows with t == 0 skipped, others land at (b, t-1)
    o = torch.full((B * (T - 1), d), 7.0, device=cuda)
    _gemm(lib, _lib, lib.dss_op_gemm_f16, A, Wt, bias, o, _lib.EPI_DROPCLS_F32, None, T, T - 1)
    want = acc.view(B, T, d)[:, 1:].reshape(-1, d)
    assert (o - want).abs().max().item() <= 2e-4 * acc.abs().max().item()
    # patch remap: row m=(b,n) -> (b, n+1) plus aux[n+1]; CLS rows untouched
    Np = T - 1
    Ap = A[: B * Np].contiguous()
    accp = Ap.float() @ Wt.float().T + bias
    pos = torch.randn(T, d, device=cuda, generator=g)
    xo = torch.full((B * T, d), 3.0, device=cuda)
    _gemm(lib, _lib, lib.dss_op_gemm_f16, Ap, Wt, bias, xo, _lib.EPI_PATCH_F32, pos, Np, T)
    want = torch.full((B, T, d), 3.0, device=cuda)
    want[:, 1:] = accp.view(B, Np, d) + pos[1:]
    assert (xo.view(B, T, d) - want).abs().max().item() <= 2e-4 * accp.abs().max().item()
    # residual f32 with K >= 1024 (the CTA-pair MMA path), one N per tile width: 128, 192, 256
    K2 = 1536
    A2 = torch.randn(M, K2, device=cuda, generator=g).half()
    for N2 in (128, 384, 768):
        W2 = (torch.randn(N2, K2, device=cuda, generator=g) * 0.05).half()
        b2 = torch.randn(N2, device=cuda, generator=g)
        acc2 = A2.float() @ W2.float().T + b2
        x = torch.randn(M, N2, device=cuda, generator=g)
        x0 = x.clone()
        _gemm(lib, _lib, lib.dss_op_gemm_f16, A2, W2, b2, x, _lib.EPI_BIAS_RESID_F32)
        assert (x - (x0 + acc2)).abs().max().item() <= 2e-4 * acc2.abs().max().item(), N2


def test_gemm_ln_and_attention_on_a_second_device(cuda):
    """A GEMM, a fused-LayerNorm GEMM and an attention call on cuda:0 and then on cuda:1 in the same process: the
    launch set-up the library keeps per device (dynamic shared-memory limit, SM count) is in place on both."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    _lib = load_pkg("_lib"); lib = _lib.load()
    M, K, N = 300, 384, 1152
    B, T, heads = 2, 197, 6
    for dev in (torch.device("cuda:0"), torch.device("cuda:1")):
        with torch.cuda.device(dev):
            g = torch.Generator(device=dev).manual_seed(11)
            st = _lib.stream_ptr(dev)
            x = torch.randn(M, K, device=dev, generator=g) * 2.0 + 0.5
            gamma = torch.randn(K, device=dev, generator=g) * 0.5 + 1.0
            beta = torch.randn(K, device=dev, generator=g) * 0.2
            Wt = (torch.randn(N, K, device=dev, generator=g) * 0.05).half()
            bias = torch.randn(N, device=dev, generator=g) * 0.1
            qkv = (torch.randn(B, T, 3 * heads * 64, device=dev, generator=g) * 1.5).half()
            A = x.half()
            out = torch.full((M, N), float("nan"), device=dev)
            out_ln = torch.full((M, N), float("nan"), device=dev, dtype=torch.float16)
            att = torch.full((B, T, heads * 64), float("nan"), device=dev, dtype=torch.float16)
            _lib.check(lib.dss_op_gemm_f16(A.data_ptr(), Wt.data_ptr(), bias.data_ptr(), out.data_ptr(), M, N, K,
                                           _lib.EPI_BIAS_F32, None, 0, 0, st), "gemm")
            _lib.check(lib.dss_op_gemm_ln_f16(x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), Wt.data_ptr(), bias.data_ptr(),
                                              out_ln.data_ptr(), M, N, K, 1e-6, 0, st), "gemm_ln")
            _lib.check(lib.dss_op_attention_tc_f16(qkv.data_ptr(), att.data_ptr(), B, T, heads, st), "attention")
            torch.cuda.synchronize(dev)
            ref = A.float() @ Wt.float().T + bias
            assert (out - ref).abs().max().item() <= 2e-4 * max(1.0, ref.abs().max().item()), dev
            xn = torch.nn.functional.layer_norm(x, (K,), gamma, beta, 1e-6)
            ref = xn.half().float() @ Wt.float().T + bias
            assert (out_ln.float() - ref).abs().max().item() <= 3e-3 * max(1.0, ref.abs().max().item()), dev
            q, k, v = qkv.float().view(B, T, 3, heads, 64).permute(2, 0, 3, 1, 4)
            ref = (((q @ k.transpose(-2, -1)) * 0.125).softmax(-1) @ v).transpose(1, 2).reshape(B, T, heads * 64)
            assert (att.float() - ref).abs().max().item() <= 4e-3 * max(1.0, ref.abs().max().item()), dev


@pytest.mark.parametrize("d", [384, 768])
def test_layernorm(cuda, d):
    _lib = load_pkg("_lib"); lib = _lib.load()
    g = torch.Generator(device="cuda").manual_seed(d)
    M = 1000
    x = torch.randn(M, d, device=cuda, generator=g) * 3 + 0.5
    gamma = torch.randn(d, device=cuda, generator=g)
    beta = torch.randn(d, device=cuda, generator=g)
    y = torch.empty(M, d, device=cuda, dtype=torch.float16)
    _lib.check(lib.dss_op_layernorm_f16(x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), y.data_ptr(), M, d, 1e-6,
                                        _lib.stream_ptr()))
    torch.cuda.synchronize()
    ref = torch.nn.functional.layer_norm(x, (d,), gamma, beta, 1e-6)
    err = (y.float() - ref).abs().max().item()
    assert err <= 1e-3 * ref.abs().max().item() + 1e-3, err   # fp16 output rounding only


@pytest.mark.parametrize("impl", ["dss_op_attention_tc_f16", "dss_op_attention_f16"])
@pytest.mark.parametrize("B,T,heads", [(1, 64, 6), (2, 197, 6), (2, 901, 6), (1, 130, 12), (3, 257, 6), (4, 577, 6),
                                       (40, 901, 6), (30, 257, 6), (70, 100, 6)])
def test_attention(cuda, B, T, heads, impl):
    _lib = load_pkg("_lib"); lib = _lib.load()
    g = torch.Generator(device="cuda").manual_seed(T)
    d = heads * 64
    qkv = (torch.randn(B, T, 3 * d, device=cuda, generator=g) * 1.5).half()
    out = torch.full((B, T, d), float("nan"), device=cuda, dtype=torch.float16)
    _lib.check(getattr(lib, impl)(qkv.data_ptr(), out.data_ptr(), B, T, heads, _lib.stream_ptr()))
    torch.cuda.synchronize()
    q, k, v = qkv.float().view(B, T, 3, heads, 64).permute(2, 0, 3, 1, 4)
    att = ((q @ k.transpose(-2, -1)) * 0.125).softmax(-1)
    ref = (att @ v).transpose(1, 2).reshape(B, T, d)
    assert torch.isfinite(out.float()).all()
    err = (out.float() - ref).abs().max().item()
    print(f"{impl} B={B} T={T}: max err {err:.3e} (ref max {ref.abs().max().item():.3f})")
    assert err <= 4e-3 * max(1.0, ref.abs().max().item()), err  # P and output rounded to fp16


@pytest.mark.parametrize("P,H,W", [(16, 224, 224), (16, 250, 333), (8, 64, 72)])
def test_im2col(cuda, P, H, W):
    _lib = load_pkg("_lib"); lib = _lib.load()
    from oracle import dino_vit
    g = torch.Generator().manual_seed(H)
    B = 2
    img = torch.randint(0, 256, (B, H, W, 3), generator=g, dtype=torch.uint8)
    Hp, Wp = H // P, W // P
    out = torch.empty(B * Hp * Wp, 3 * P * P, device=cuda, dtype=torch.float16)
    img_d = img.to(cuda)
    _lib.check(lib.dss_op_im2col_f16(img_d.data_ptr(), out.data_ptr(), B, H, W, P, _lib.stream_ptr()))
    torch.cuda.synchronize()
    for b in range(B):
        x = dino_vit.preprocess_u8(img[b], P)  # (1,3,Hc,Wc)
        ref = torch.nn.functional.unfold(x, kernel_size=P, stride=P)[0].T  # (Np, 3*P*P), (c,py,px) order
        got = out[b * Hp * Wp:(b + 1) * Hp * Wp].float().cpu()
        assert (got - ref).abs().max().item() <= 2e-3
