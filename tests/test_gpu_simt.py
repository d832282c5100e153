"""GPU: the FFMA (fp32 verification mode) convolution and attention kernels against torch fp32."""
import math

import pytest
import torch
import torch.nn.functional as Fn

pytestmark = pytest.mark.gpu


def _conv_ref(x_nhwc, w, b, stride, row_add=None, residual=None, x2=None, w2=None):
    y = Fn.conv2d(x_nhwc.float().permute(0, 3, 1, 2), w.float(), b, stride=stride, padding=w.shape[-1] // 2)
    if x2 is not None:
        y = y + Fn.conv2d(x2.float().permute(0, 3, 1, 2), w2.float())
    if row_add is not None:
        y = y + row_add[:, :, None, None]
    if residual is not None:
        y = y + residual.float().permute(0, 3, 1, 2)
    return y


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("B,H,W,Cin,Cout,ks,stride", [(2, 16, 16, 64, 64, 3, 1), (1, 8, 8, 128, 192, 3, 1),
                                                      (3, 16, 8, 32, 48, 1, 1), (2, 16, 16, 64, 64, 3, 2),
                                                      (1, 32, 32, 16, 6, 3, 1), (2, 5, 7, 16, 80, 3, 1)])
def test_conv_simt(cuda_lib, dtype, B, H, W, Cin, Cout, ks, stride):
    from fidm_b200 import ops
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    dev = "cuda"
    g = torch.Generator(device=dev).manual_seed(B * 100 + Cin)
    x = torch.randn(B, H, W, Cin, device=dev, generator=g).to(dtype)
    w = (torch.randn(Cout, Cin, ks, ks, device=dev, generator=g) / math.sqrt(Cin * ks * ks)).to(dtype)
    b = torch.randn(Cout, device=dev, generator=g)
    wk = ops.repack_weight(w.float(), dtype)
    tol = dict(atol=1e-4, rtol=1e-4) if dtype == torch.float32 else dict(atol=3e-2, rtol=2e-2)
    y = ops.conv2d(x, wk, b, stride=stride, impl="simt")
    want = _conv_ref(x, w, b, stride)
    assert torch.allclose(y.float().permute(0, 3, 1, 2), want, **tol)
    if stride == 1:
        Ho, Wo = want.shape[2:]
        row = torch.randn(B, Cout + 8, device=dev, generator=g)[:, 4:4 + Cout]
        res = torch.randn(B, Ho, Wo, Cout, device=dev, generator=g).to(dtype)
        x2 = torch.randn(B, Ho, Wo, 32, device=dev, generator=g).to(dtype)
        w2 = (torch.randn(Cout, 32, 1, 1, device=dev, generator=g) / math.sqrt(32)).to(dtype)
        y = ops.conv2d(x, wk, b, row_add=row, residual=res, x2=x2, w2=ops.repack_weight(w2.float(), dtype), impl="simt")
        want = _conv_ref(x, w, b, 1, row, res, x2, w2)
        assert torch.allclose(y.float().permute(0, 3, 1, 2), want, **tol)
        yn = ops.conv2d(x, wk, b, nchw_out_channels=min(Cout, 6), impl="simt")
        assert torch.allclose(yn, _conv_ref(x, w, b, 1)[:, :min(Cout, 6)], **tol)


@pytest.fixture(scope="module")
def simt_report(request):
    """(kernel, dtype) -> largest error / bound of test_attention_simt, written to the terminal after the module."""
    rows = {}
    yield rows
    tr = request.config.pluginmanager.get_plugin("terminalreporter")
    if tr is not None and rows:
        with request.config.pluginmanager.get_plugin("capturemanager").global_and_fixture_disabled():
            tr.write_line("")
            for (kernel, dtype), ratio in sorted(rows.items()):
                tr.write_line(f"SIMT attention {kernel} {dtype}: max error/bound {ratio:.3f}")


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("B,T,heads,d", [(2, 64, 4, 64), (1, 256, 4, 64), (2, 64, 4, 128), (1, 100, 2, 32),
                                         (1, 1024, 2, 64), (2, 100, 3, 16),
                                         # head dims outside the tiled kernel's set (nn.py:245-249: d = C / heads is free):
                                         (2, 64, 2, 96), (1, 100, 3, 48), (1, 256, 1, 256), (1, 64, 1, 1024), (2, 70, 2, 20)])
def test_attention_simt(cuda_lib, simt_report, dtype, B, T, heads, d):
    """Random inputs against `simt_error_bound` (float64 reference); the gather construction exactly (each query
    selects one key by >= 32 logits); every valid key at the same negative logit, with the padding keys of a partial
    tile (score 0 if they were counted) masked."""
    from fidm_b200 import ops
    from oracle import attention_oracle as ao
    kernel = "tiled" if d in (16, 32, 64, 128) else "generic"
    qkv = ao.random_qkv(B, T, heads, d, seed=T + d, scale=1.5, dtype=dtype, device="cuda")
    y = ops.attention(qkv, heads, impl="simt")
    ref, w = ao.attention_f64(qkv, heads)
    ratio = ((y.double() - ref).abs() / ao.simt_error_bound(w, qkv[..., 2 * heads * d:], ref, dtype)).max().item()

    qkv, expected, _ = ao.gather(B, T, heads, d, seed=T + d, dtype=dtype, device="cuda")
    y = ops.attention(qkv, heads, impl="simt")
    assert torch.equal(y, expected), f"gather: {(y != expected).sum().item()} elements differ"

    qkv, expected = ao.uniform_negative(B, T, heads, d, seed=T + d, dtype=dtype, device="cuda")
    y = ops.attention(qkv, heads, impl="simt")
    tol = ao.uniform_negative_bound(qkv, expected, out_rel=ao.U_BF16 if dtype == torch.bfloat16 else 2.0 ** -24)
    ratio_u = ((y.double() - expected).abs() / tol).max().item()
    key = (kernel, str(dtype).replace("torch.", ""))
    simt_report[key] = max(simt_report.get(key, 0.0), ratio, ratio_u)
    assert ratio <= 1.0, ratio
    assert ratio_u <= 1.0, ratio_u
