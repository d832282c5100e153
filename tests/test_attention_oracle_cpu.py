"""CPU: the attention oracle (oracle/attention_oracle.py) -- its constructions have the properties the GPU tests rely
on, a CPU emulation of K3's arithmetic (csrc/attention_tc.cu) stays inside `tc_error_bound` at every shipped shape,
and emulations with one deliberate K3 mistake each fail the check that targets that mistake.  This shows without a
GPU that the assertions of tests/test_gpu_attention_tc.py are neither flaky nor toothless."""
import math

import pytest
import torch
import torch.nn.functional as Fn

from helpers import attention_shapes
from oracle import attention_oracle as ao

BK = 128                          # K3's key tile
SHIPPED = {"ADM256": {(1024, 8, 64), (256, 16, 64), (64, 16, 64)},
           "REF_FFHQ256": {(256, 8, 64), (64, 8, 64)},
           "T64": {(256, 4, 64), (64, 4, 128)}}
SHAPES = sorted(set().union(*SHIPPED.values()))
SCALES = (0.5, 1.0, 1.5)         # logits of standard deviation 0.25, 1 and 2.25
BATCHES = (1, 2, 8)
MUTATIONS = ("no_rescale", "last_tile_mask_off_by_one", "padding_counted", "v_subtiles_swapped")


def emulate_k3(qkv, heads, mutation=None):
    """K3's arithmetic on the CPU: 128-key tiles, fp32 scores, online row maximum, p = exp2(fma(s, c, -m c)) in
    fp32 with c = fp32(d^-1/2 * log2 e) as the host computes it, P rounded to bf16 for the PV product, l summed
    from the unrounded p, O and l rescaled by alpha = exp2((m_old - m_new) c), out = bf16(O * (1 / l)).
    `mutation` plants one mistake (see MUTATIONS)."""
    q, k, v = (x.float() for x in ao.split_heads(qkv, heads))
    n, h, t, d = q.shape
    if mutation == "v_subtiles_swapped":            # the two 64-channel sub-tiles of V exchanged (d = 128)
        v = torch.cat([v[..., 64:], v[..., :64]], dim=-1)
    if mutation == "padding_counted":               # the zero-filled keys past t take part like valid ones
        pad = -t % BK
        k, v = Fn.pad(k, (0, 0, 0, pad)), Fn.pad(v, (0, 0, 0, pad))
    c = torch.tensor(1.0) / torch.sqrt(torch.tensor(float(d))) * torch.tensor(1.4426950408889634)
    s = torch.matmul(q, k.transpose(-1, -2))
    m = torch.full((n, h, t), -math.inf)
    l = torch.zeros(n, h, t)
    o = torch.zeros(n, h, t, d)
    for j0 in range(0, s.shape[-1], BK):
        kv = min(BK, s.shape[-1] - j0)
        if mutation == "last_tile_mask_off_by_one":   # min(BK, T - j*BK - 1): the last valid key is dropped
            kv = min(BK, t - j0 - 1)
        st = s[..., j0:j0 + kv]
        m_new = torch.maximum(m, st.amax(-1))
        alpha = torch.exp2((m - m_new) * c)
        if mutation == "no_rescale" and j0 > 0:
            alpha = torch.ones_like(alpha)
        mb = m_new * c
        p = torch.exp2((st.double() * c.double() - mb.double()[..., None]).float())     # fmaf(s, c, -mb)
        l = l * alpha + p.sum(-1)
        o = o * alpha[..., None] + torch.matmul(p.bfloat16().float(), v[..., j0:j0 + kv, :])
        m = m_new
    return ao.merge_heads((o * (1.0 / l)[..., None]).bfloat16())


def bound_ratio(y, ref, bound):
    return ((y.double() - ref).abs() / bound).max().item()


def rel_l2(y, ref):
    return ((y.double() - ref).norm() / ref.norm()).item()


def random_case(shape, scale, batch=1):
    """The random inputs of tests/test_gpu_attention_tc.py::test_shipped_shapes (same seeds), their float64
    reference and bound."""
    t, heads, d = shape
    qkv = ao.random_qkv(batch, t, heads, d, seed=1000 * batch + t + heads + d, scale=scale)
    ref, w = ao.attention_f64(qkv, heads)
    return qkv, ref, ao.tc_error_bound(w, qkv[..., 2 * heads * d:], ref)


def test_shipped_attention_shapes():
    """Every (tokens, heads, head_dim) K3 runs in the shipped plans, derived from the model configurations."""
    from fidm_b200.arch import CONFIGS
    assert {name: attention_shapes(cfg) for name, cfg in CONFIGS.items()} == SHIPPED


@pytest.mark.parametrize("t,d,dtype", [(1, 64, torch.bfloat16), (64, 64, torch.bfloat16), (100, 128, torch.bfloat16),
                                       (1024, 64, torch.bfloat16), (4096, 128, torch.bfloat16),
                                       (70, 20, torch.float32), (100, 48, torch.float32), (64, 16, torch.float32),
                                       (256, 256, torch.float32), (1024, 64, torch.float32)])
def test_gather_properties(t, d, dtype):
    n, heads = (1, 1) if t > 1024 else (2, 2)
    qkv, expected, perm = ao.gather(n, t, heads, d, seed=t + d, dtype=dtype)
    ref, w = ao.attention_f64(qkv, heads)
    assert torch.equal(ref.to(dtype), expected)                     # exact in the storage type
    assert torch.equal(perm.sort(-1).values, torch.arange(t).expand_as(perm))   # each key answers exactly one query
    others = w.clone()
    others.scatter_(-1, perm[..., None], 0.0)
    assert others.amax().item() < 1.3e-14 and others.sum(-1).amax().item() < ao.code_bits(t) * 1.3e-14
    q, k, _ = ao.split_heads(qkv, heads)
    logits = torch.matmul(q.double(), k.double().transpose(-1, -2)) / math.sqrt(d)
    top2 = logits.topk(min(2, t), dim=-1).values
    if t > 1:
        assert (top2[..., 0] - top2[..., 1]).amin().item() >= 32.0
    if t >= 64:    # exp2(logit * log2 e) overflows fp32 unless the running maximum is subtracted
        assert logits.amax().item() * math.log2(math.e) > 128.0
    if dtype == torch.bfloat16 and d in (64, 128):
        assert torch.equal(emulate_k3(qkv, heads), expected)


@pytest.mark.parametrize("t,d", [(64, 64), (192, 64), (1024, 64), (192, 128), (1000, 128)])
def test_uniform_negative_properties(t, d):
    qkv, expected = ao.uniform_negative(2, t, 2, d, seed=t)
    q, k, _ = ao.split_heads(qkv, 2)
    logits = torch.matmul(q.double(), k.double().transpose(-1, -2)) / math.sqrt(d)
    assert torch.equal(logits, torch.full_like(logits, -64.0 / math.sqrt(d)))
    ref, _ = ao.attention_f64(qkv, 2)
    assert torch.allclose(ref, expected, rtol=1e-12, atol=1e-14)
    assert bound_ratio(emulate_k3(qkv, 2), expected, ao.uniform_negative_bound(qkv, expected)) <= 1.0


@pytest.mark.parametrize("kind", ao.RAMP_KINDS)
@pytest.mark.parametrize("t,d", [(64, 64), (192, 64), (1024, 64), (192, 128), (1000, 128)])
def test_ramp_properties(kind, t, d):
    heads = 2
    qkv = ao.ramp(2, t, heads, d, seed=t + d, kind=kind)
    q, k, _ = ao.split_heads(qkv, heads)
    logits = torch.matmul(q.double(), k.double().transpose(-1, -2)) / math.sqrt(d)
    tile_max = torch.stack([logits[..., j0:j0 + BK].amax(-1) for j0 in range(0, t, BK)], dim=-1)
    if kind == "rising":          # alpha < 1 at every tile boundary, every row
        assert (tile_max.diff(dim=-1) > 0.25).all()
    elif kind == "falling":       # the maximum never moves after the first tile
        assert (tile_max[..., 1:] < tile_max[..., :1]).all()
    else:                         # the maximum arrives in the last tile, the other keys keep a real share
        assert (tile_max[..., -1:] > tile_max[..., :-1] + 2.0).all()
        w_spike = torch.softmax(logits, -1).amax(-1)
        assert w_spike.amin().item() > 0.2 and w_spike.amax().item() < 0.8
    ref, w = ao.attention_f64(qkv, heads)
    bound = ao.tc_error_bound(w, qkv[..., 2 * heads * d:], ref)
    assert bound_ratio(emulate_k3(qkv, heads), ref, bound) <= 0.7


@pytest.mark.parametrize("shape", SHAPES)
def test_emulation_within_bound(shape):
    """The bound is not flaky: on the GPU test's inputs, emulated K3 arithmetic stays at or below 0.7 of it, and
    rel-L2 below 3e-3 (the GPU test allows 4e-3)."""
    for batch in BATCHES:
        for scale in SCALES:
            qkv, ref, bound = random_case(shape, scale, batch)
            y = emulate_k3(qkv, shape[1])
            assert bound_ratio(y, ref, bound) <= 0.7, (batch, scale)
            assert rel_l2(y, ref) < 3e-3, (batch, scale)


@pytest.mark.parametrize("mutation", MUTATIONS)
def test_mutations_fail(mutation):
    """The bound is not toothless: each planted mistake fails the check that targets it by a wide margin."""
    if mutation == "no_rescale":
        for shape in [s for s in SHAPES if s[0] >= 192]:
            qkv, ref, bound = random_case(shape, 1.5)
            assert bound_ratio(emulate_k3(qkv, shape[1], mutation), ref, bound) > 100, shape
        for t in (192, 1024):
            qkv = ao.ramp(1, t, 2, 64, seed=t, kind="rising")
            ref, w = ao.attention_f64(qkv, 2)
            assert bound_ratio(emulate_k3(qkv, 2, mutation), ref, ao.tc_error_bound(w, qkv[..., 256:], ref)) > 10
    elif mutation == "last_tile_mask_off_by_one":
        for t, d in ((64, 64), (100, 128), (1024, 64)):
            qkv, expected, _ = ao.gather(2, t, 2, d, seed=t + d)
            assert not torch.equal(emulate_k3(qkv, 2, mutation), expected), (t, d)
        for shape in SHAPES:
            qkv, ref, bound = random_case(shape, 1.5)
            assert bound_ratio(emulate_k3(qkv, shape[1], mutation), ref, bound) > 10, shape
    elif mutation == "padding_counted":
        for t, d in ((64, 64), (192, 64), (192, 128), (1000, 128)):
            qkv, expected = ao.uniform_negative(2, t, 2, d, seed=t)
            y = emulate_k3(qkv, 2, mutation)
            assert bound_ratio(y, expected, ao.uniform_negative_bound(qkv, expected)) > 100, (t, d)
    else:
        qkv, expected, _ = ao.gather(2, 64, 4, 128, seed=1)
        assert not torch.equal(emulate_k3(qkv, 4, mutation), expected)
        qkv, ref, bound = random_case((64, 4, 128), 1.5)
        assert bound_ratio(emulate_k3(qkv, 4, mutation), ref, bound) > 100
