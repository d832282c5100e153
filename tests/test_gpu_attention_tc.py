"""GPU: K3 (attn_tc_kernel, csrc/attention_tc.cu) against a float64 reference of nn.py:222-235.

Every comparison is either exact (inputs whose answer is exact in bf16, and bitwise invariants between runs) or
against `tc_error_bound`, an elementwise bound derived from where K3 rounds (oracle/attention_oracle.py).
tests/test_attention_oracle_cpu.py shows on the CPU that an emulation of K3's arithmetic stays at or below 0.7 of
that bound on the inputs used here, and that each planted mistake (no rescale, a mask off by one, padding keys
counted, swapped V sub-tiles) fails it.  The largest error / bound ratio and rel-L2 of each group are written to the
terminal at the end of the module.
"""
import ctypes as C

import pytest
import torch

from helpers import attention_shapes
from oracle import attention_oracle as ao

pytestmark = pytest.mark.gpu

E_BADARG, E_SHAPE, E_ALIGN = -1, -2, -3          # include/fidm_b200.h


def _shipped_shapes():
    from fidm_b200.arch import CONFIGS
    return sorted(set().union(*(attention_shapes(cfg) for cfg in CONFIGS.values())))


SHIPPED = _shipped_shapes()          # (tokens, heads, head_dim); the table is pinned by test_attention_oracle_cpu.py
SCALES = (0.5, 1.0, 1.5)
SENTINEL = -12345.0                  # no attention output reaches it (|out| <= max |v|)


def _shape_id(shape):
    return "T%d-h%d-d%d" % shape


@pytest.fixture(scope="module")
def report(request):
    """group -> (largest error / bound, largest rel-L2), written to the terminal after the module."""
    rows = {}
    yield rows
    lines = [f"K3 {group}: max error/bound {ratio:.3f}" + ("" if rel is None else f", rel-L2 {rel:.2e}")
             for group, (ratio, rel) in sorted(rows.items())]
    _write_terminal(request.config, lines)


def _write_terminal(config, lines):
    """Past output capture, so that the figures show in a -q run that passes."""
    tr = config.pluginmanager.get_plugin("terminalreporter")
    if tr is None or not lines:
        return
    with config.pluginmanager.get_plugin("capturemanager").global_and_fixture_disabled():
        tr.write_line("")
        for line in lines:
            tr.write_line(line)


def _record(report, group, ratio, rel=None):
    r0, l0 = report.get(group, (0.0, None))
    report[group] = (max(r0, ratio), l0 if rel is None else max(rel, l0 or 0.0))


def _tc(qkv, heads, out=None):
    from fidm_b200 import ops
    y = ops.attention(qkv, heads, out=out, impl="tc")
    torch.cuda.synchronize()
    return y


def _check_bound(report, group, qkv, heads, y, max_rel=None):
    ref, w = ao.attention_f64(qkv, heads)
    bound = ao.tc_error_bound(w, qkv[..., 2 * (qkv.shape[-1] // 3):], ref)
    err = (y.double() - ref).abs()
    ratio = (err / bound).max().item()
    rel = ((y.double() - ref).norm() / ref.norm()).item()
    _record(report, group, ratio, rel)
    bad = (err > bound).sum().item()
    assert bad == 0, f"{bad} elements outside the bound, max error/bound {ratio:.3g}"
    if max_rel is not None:
        assert rel < max_rel, rel


@pytest.mark.parametrize("d", [64, 128])
@pytest.mark.parametrize("B,T,heads", [(1, 128, 1), (2, 64, 4), (1, 256, 8), (2, 1024, 8), (3, 192, 2)])
def test_attention_tc(cuda_lib, report, B, T, heads, d):
    """head dims 64 and 128 (num_heads-defined heads of 512-channel blocks, nn.py:245-249), read through a strided
    view of a wider buffer"""
    buf = ao.random_qkv(B, T, heads, d, seed=T + heads + d, scale=1.5).cuda()
    buf = torch.cat([torch.zeros_like(buf[..., :64]), buf], dim=-1)
    qkv = buf[..., 64:]
    _check_bound(report, "strided random", qkv, heads, _tc(qkv, heads), max_rel=4e-3)


@pytest.mark.parametrize("batch", [1, 2, 8])
@pytest.mark.parametrize("shape", SHIPPED, ids=_shape_id)
def test_shipped_shapes(cuda_lib, report, shape, batch):
    """The (T, heads, d) of every attention layer of the shipped configurations, at the benchmarked batch sizes.
    Same inputs (seeds) as test_attention_oracle_cpu.py::test_emulation_within_bound."""
    t, heads, d = shape
    for scale in SCALES:
        qkv = ao.random_qkv(batch, t, heads, d, seed=1000 * batch + t + heads + d, scale=scale, device="cuda")
        _check_bound(report, f"shipped {shape}", qkv, heads, _tc(qkv, heads), max_rel=4e-3)


@pytest.mark.parametrize("d", [64, 128])
@pytest.mark.parametrize("t", [64, 100, 256, 1024, 4096])
def test_gather_exact(cuda_lib, t, d):
    """Each query selects one key by a margin of >= 32 logits, its largest logit overflowing exp2 unless the running
    maximum is subtracted: the output is exactly that key's v row, bit for bit, for every (image, head, query)."""
    qkv, expected, _ = ao.gather(2, t, 3, d, seed=t + d, device="cuda")
    y = _tc(qkv, 3)
    assert torch.equal(y, expected), f"{(y != expected).sum().item()} elements differ"


@pytest.mark.parametrize("d", [64, 128])
@pytest.mark.parametrize("t", [64, 192, 1024])
def test_uniform_negative(cuda_lib, report, t, d):
    """All valid keys score the same negative logit; a padding key taken into the row (score 0) would dominate."""
    qkv, expected = ao.uniform_negative(2, t, 2, d, seed=t, device="cuda")
    y = _tc(qkv, 2)
    ratio = ((y.double() - expected).abs() / ao.uniform_negative_bound(qkv, expected)).max().item()
    _record(report, "uniform-negative", ratio)
    assert ratio <= 1.0, ratio


@pytest.mark.parametrize("kind", ao.RAMP_KINDS)
@pytest.mark.parametrize("d", [64, 128])
@pytest.mark.parametrize("t", [64, 192, 1024])
def test_ramps(cuda_lib, report, t, d, kind):
    """The row maximum moves into every new key tile (rising), never moves (falling), or jumps at the last tile."""
    qkv = ao.ramp(2, t, 2, d, seed=t + d, kind=kind, device="cuda")
    _check_bound(report, f"ramp {kind}", qkv, 2, _tc(qkv, 2))


@pytest.mark.parametrize("d", [64, 128])
@pytest.mark.parametrize("t", [1, 65, 100, 129, 200, 1000])
def test_partial_tiles(cuda_lib, report, t, d):
    """Token counts that leave a partial 128-query and 128-key tile.  The engine sends K3 only T % 64 == 0, but the
    C ABI accepts any T."""
    qkv = ao.random_qkv(2, t, 2, d, seed=t + d, device="cuda")
    _check_bound(report, "partial-tile random", qkv, 2, _tc(qkv, 2), max_rel=4e-3)
    qkv, expected, _ = ao.gather(2, t, 2, d, seed=t + d + 1, device="cuda")
    y = _tc(qkv, 2)
    assert torch.equal(y, expected), f"gather: {(y != expected).sum().item()} elements differ"


@pytest.mark.parametrize("shape", SHIPPED, ids=_shape_id)
def test_bitwise_invariants(cuda_lib, shape):
    """Each CTA owns one (image, head, 128 queries) and reduces in a fixed order, so the result of an image must not
    depend on the batch around it, the order of the heads, the row stride of qkv or the run."""
    t, heads, d = shape
    c = heads * d
    qkv = ao.random_qkv(8, t, heads, d, seed=t + heads + d, device="cuda")
    y = _tc(qkv, heads)
    for b in range(8):
        assert torch.equal(_tc(qkv[b:b + 1].clone(), heads), y[b:b + 1]), f"image {b} alone"
    assert torch.equal(_tc(qkv, heads), y), "second run"
    perm = torch.randperm(heads, generator=torch.Generator().manual_seed(t)).cuda()
    qkv_p = qkv.reshape(8, t, 3, heads, d)[:, :, :, perm].reshape(8, t, 3 * c)
    assert torch.equal(_tc(qkv_p, heads), y.reshape(8, t, heads, d)[:, :, perm].reshape(8, t, c)), "heads permuted"
    wide = torch.full((8, t, 3 * c + 192), SENTINEL, device="cuda", dtype=torch.bfloat16)
    wide[..., 128:128 + 3 * c] = qkv
    assert torch.equal(_tc(wide[..., 128:128 + 3 * c], heads), y), "ld_qkv = 3C + 192"
    if shape == (1024, 8, 64):
        qkv32 = ao.random_qkv(32, t, heads, d, seed=32, device="cuda")
        y32 = _tc(qkv32, heads)
        for b in (0, 13, 31):
            assert torch.equal(_tc(qkv32[b:b + 1].clone(), heads), y32[b:b + 1]), f"image {b} of 32 alone"


@pytest.mark.parametrize("d", [64, 128])
@pytest.mark.parametrize("t", [64, 200, 1000])
def test_output_bounds(cuda_lib, t, d):
    """K3 writes only its [N, T, C] output: into a channel slice of a wider sentinel-filled buffer with one more image
    after it, nothing outside the slice changes (including the rows past T of a partial last query tile)."""
    n, heads = 2, 2
    c = heads * d
    qkv = ao.random_qkv(n, t, heads, d, seed=t + d, device="cuda")
    want = _tc(qkv, heads)
    buf = torch.full((n + 1, t, c + 128), SENTINEL, device="cuda", dtype=torch.bfloat16)
    _tc(qkv, heads, out=buf[:n, :, 64:64 + c])
    assert torch.equal(buf[:n, :, 64:64 + c], want)
    buf[:n, :, 64:64 + c] = SENTINEL
    assert (buf == SENTINEL).all(), f"{(buf != SENTINEL).sum().item()} elements outside the output changed"


def _call(qkv, out, heads, head_dim=None, ld_qkv=None, ld_out=None):
    """fidm_attention_qkv_nhwc_bf16 with explicit arguments (ops.attention derives them from the tensors)."""
    from fidm_b200 import _lib as L
    n, t, c3 = qkv.shape
    a = L.AttnArgs()
    a.dtype, a.batch, a.tokens, a.heads = L.dtype_code(qkv.dtype), n, t, heads
    a.head_dim = head_dim or c3 // 3 // heads
    a.qkv, a.ld_qkv = L.ptr(qkv), ld_qkv or qkv.stride(1)
    a.out, a.ld_out = L.ptr(out), ld_out or out.stride(1)
    L.check(L.lib().fidm_attention_qkv_nhwc_bf16(C.byref(a), L.stream()), "attention/tc")


def test_rejections(cuda_lib):
    """Arguments K3 cannot take are refused on the host, with the code the caller dispatches on, before any launch:
    the output keeps its sentinel."""
    from fidm_b200._lib import ArgumentError
    n, t, heads, d = 2, 128, 2, 64
    c = heads * d

    def qkv_in(width, dtype=torch.bfloat16):
        return torch.randn(n, t, width, device="cuda").to(dtype)

    def out_in(width):
        return torch.full((n, t, width), SENTINEL, device="cuda", dtype=torch.bfloat16)

    cases = [  # (what, qkv, out, heads, extra arguments, code)
        ("head_dim 32", qkv_in(3 * 4 * 32), out_in(4 * 32), 4, {}, E_SHAPE),
        ("head_dim 96", qkv_in(3 * 2 * 96), out_in(2 * 96), 2, {}, E_SHAPE),
        ("fp32", qkv_in(3 * c, torch.float32), out_in(c), heads, {}, E_BADARG),
        ("ld_qkv < 3C", qkv_in(3 * c), out_in(c), heads, dict(ld_qkv=3 * c - 8), E_BADARG),
        ("ld_out < C", qkv_in(3 * c), out_in(c), heads, dict(ld_out=c - 8), E_BADARG),
        ("qkv base + 8 bytes", qkv_in(3 * c + 8)[..., 4:4 + 3 * c], out_in(c), heads, {}, E_ALIGN),
        ("out base + 8 bytes", qkv_in(3 * c), out_in(c + 8)[..., 4:4 + c], heads, {}, E_ALIGN),
        ("ld_qkv % 8 == 4", qkv_in(3 * c + 4)[..., :3 * c], out_in(c), heads, {}, E_ALIGN),
        ("ld_out % 8 == 4", qkv_in(3 * c), out_in(c + 4)[..., :c], heads, {}, E_ALIGN),
    ]
    for what, qkv, out, h, extra, code in cases:
        with pytest.raises(ArgumentError, match=rf"\(code {code}\)$"):
            _call(qkv, out, h, **extra)
        torch.cuda.synchronize()
        assert (out == SENTINEL).all(), what
