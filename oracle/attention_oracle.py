"""CPU ORACLE (test infrastructure only) -- QKV attention.

Checker only: imported by `tests/`, never by the product path.  Plain torch on whatever device the input lives on.

  * `attention_f64`: the operation of nn.py:222-235 (QKVAttention) on an NHWC-flattened `[N, T, 3C]` buffer whose
    channel order is [Q heads | K heads | V heads], in float64 from the stored values; it also returns the softmax
    weights W, which the error bounds need;
  * `tc_error_bound` / `simt_error_bound`: elementwise bounds on |kernel - float64| derived from where each kernel
    rounds (derivations in the docstrings);
  * input constructions that make specific kernel mistakes visible: `gather` (an exact expected output, every key
    the winner of exactly one query), `uniform_negative` (every valid key scores the same negative logit, so a
    zero-filled padding key would outweigh it) and `ramp` (the running maximum moves from key tile to key tile).

Every construction draws from a seeded CPU generator and then moves to `device`, so the same seed gives the same
input on every device.
"""
import math

import torch

U_BF16 = 2.0 ** -8          # unit roundoff of bfloat16 (8 significand bits, round to nearest)


def split_heads(qkv, heads):
    """[N, T, 3C] -> q, k, v as [N, heads, T, d] views (head h = channels [h*d, (h+1)*d) of each third)."""
    n, t, c3 = qkv.shape
    c = c3 // 3
    d = c // heads
    return tuple(qkv[..., i * c:(i + 1) * c].reshape(n, t, heads, d).transpose(1, 2) for i in range(3))


def merge_heads(x):
    """[N, heads, T, d] -> [N, T, heads*d]."""
    n, h, t, d = x.shape
    return x.transpose(1, 2).reshape(n, t, h * d)


def attention_f64(qkv, heads, *, max_chunk_elems=1 << 24):
    """nn.py:222-235 on `qkv` [N, T, 3C]: returns (out [N, T, C], W [N, heads, T, T]), both float64.

    w = softmax((q * d^-1/4)^T (k * d^-1/4)), a = w v^T, computed from the stored (bf16 or fp32) values.  The score
    and weight temporaries are built a few images at a time (at most `max_chunk_elems` doubles each), so that at
    (N, T, heads) = (8, 1024, 8) the whole call needs W (512 MB) plus 256 MB.
    """
    n, t, _ = qkv.shape
    q, k, v = split_heads(qkv, heads)
    d = q.shape[-1]
    s = d ** -0.25
    out = torch.empty(n, heads, t, d, dtype=torch.float64, device=qkv.device)
    w_all = torch.empty(n, heads, t, t, dtype=torch.float64, device=qkv.device)
    step = max(1, max_chunk_elems // (heads * t * t))
    for b0 in range(0, n, step):
        sl = slice(b0, b0 + step)
        w = torch.matmul(q[sl].double() * s, (k[sl].double() * s).transpose(-1, -2))
        w = torch.softmax(w, dim=-1)
        w_all[sl] = w
        out[sl] = torch.matmul(w, v[sl].double())
        del w
    return merge_heads(out), w_all


def weighted_abs_v(W, V):
    """W . |V| per output element: W [N, heads, T, T], V [N, T, C] -> [N, T, C] float64."""
    n, heads, t, _ = W.shape
    vh = V.double().abs().reshape(n, t, heads, -1).transpose(1, 2)
    return merge_heads(torch.matmul(W, vh))


def error_bound(W, V, ref, p_rel, out_rel, abs_tol=1e-6):
    """p_rel (W . |V|) + out_rel |ref| + abs_tol, elementwise."""
    return p_rel * weighted_abs_v(W, V) + out_rel * ref.abs() + abs_tol


def tc_error_bound(W, V, ref):
    """Bound on |K3 - float64| elementwise: (2^-8 + 2^-10) (W . |V|) + 2^-8 |ref| + 1e-6.

    K3 (csrc/attention_tc.cu) computes, per query row, out = bf16(sum_j bf16(p_j) v_j / l) with
    p_j = exp2(s_j c - m c) relative to the running maximum m and l = sum_j p_j.
      * P is rounded to bf16 before the PV MMA: bf16(p_j) = p_j (1 + e_j), |e_j| <= u = 2^-8.  The numerator is off
        by at most u sum_j p_j |v_j|, and dividing by l (summed from the UNROUNDED fp32 p_j, so it carries no e_j)
        turns that into u (W . |V|).  Rescaling by alpha happens after the rounding and does not change e_j.
      * The output is rounded to bf16: another u |out| <= u |ref| + (higher order).
      * The fp32 scores (exact bf16 products, fp32 accumulation), the fp32 exp2 argument s c - m c, exp2f itself and
        the fp32 accumulation of O and l in TMEM / registers each contribute a relative error of a few 2^-24 per
        operation, over at most a few thousand terms: more than 10x below the P term.  The extra 2^-10 (W . |V|)
        covers all of them.
      * 1e-6 absorbs outputs that are zero up to cancellation.
    """
    return error_bound(W, V, ref, U_BF16 + 2.0 ** -10, U_BF16)


def simt_error_bound(W, V, ref, dtype):
    """Bound on |SIMT attention - float64|: 2^-12 (W . |V|) + u_out |ref| + 1e-6.

    attn_simt_kernel / attn_generic_kernel (csrc/attention_simt.cu) keep P in fp32, so the P term of
    `tc_error_bound` shrinks to the fp32 errors of the scores, expf and the accumulation, bounded here by 2^-12.
    The output is rounded once to the storage type: u_out = 2^-8 for bf16, 2^-24 for fp32.
    """
    return error_bound(W, V, ref, 2.0 ** -12, U_BF16 if dtype == torch.bfloat16 else 2.0 ** -24)


# ------------------------------------------------------------------------------------------------ constructions
def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _pack(q, k, v, dtype, device):
    """q, k, v [N, heads, T, d] (values representable in `dtype`) -> qkv [N, T, 3C]."""
    return torch.cat([merge_heads(q), merge_heads(k), merge_heads(v)], dim=-1).to(dtype).to(device)


def _round(x, dtype):
    return x.to(dtype).to(torch.float32)


def random_qkv(n, t, heads, d, seed, scale=1.0, dtype=torch.bfloat16, device="cpu"):
    """Gaussian q, k, v of standard deviation `scale` (logits of standard deviation scale^2)."""
    x = torch.randn(n, t, 3 * heads * d, generator=_gen(seed)) * scale
    return x.to(dtype).to(device)


def code_bits(t):
    """Number of code channels of `gather`: ceil(log2 t), at least 1."""
    return max(1, math.ceil(math.log2(t)))


def gather_scale(d):
    """Query amplitude of `gather`: the smallest power of two >= 16 sqrt(d) (128 at d = 64, 256 at d = 128), so
    that the best key beats every other by at least 2 a / sqrt(d) >= 32 logits."""
    return float(2 ** math.ceil(math.log2(16 * math.sqrt(d))))


def gather(n, t, heads, d, seed, dtype=torch.bfloat16, device="cpu"):
    """A query that picks exactly one key.  Returns (qkv, expected [N, T, C] in `dtype`, perm [N, heads, T]).

    nb = ceil(log2 t) code channels.  Key j holds the +-1 binary code of j in channels [0, nb) and random values in
    the others; query i holds a * code(perm(i)) in the code channels and zeros elsewhere, with perm a random
    permutation per (image, head).  Score(i, j) = a (nb - 2 hamming(perm(i), j)) / sqrt(d): the best key perm(i)
    wins by 2 a / sqrt(d) >= 32 logits (weight of any other key < e^-32 = 1.3e-14, all of them together
    < nb e^-32), and the best logit a nb / sqrt(d) overflows exp (and exp2 after the log2(e) scale) for t >= 64
    unless the running maximum is subtracted.  |v| >= 1/16, so the perturbation of the winner by the other keys is
    far below half an ulp of fp32: the exact output is v[perm(i)] in bf16 and in fp32.  Since perm is a bijection,
    every key -- the first and last of every 128-key tile and of a partial last tile included -- is the answer of
    exactly one query row.
    """
    g = _gen(seed)
    nb = code_bits(t)
    assert nb <= d, (t, d)
    a = gather_scale(d)
    bits = ((torch.arange(t)[:, None] >> torch.arange(nb)) & 1).float() * 2 - 1            # [t, nb]
    perm = torch.stack([torch.randperm(t, generator=g) for _ in range(n * heads)]).reshape(n, heads, t)
    k = torch.randn(n, heads, t, d, generator=g)
    k[..., :nb] = bits
    q = torch.zeros(n, heads, t, d)
    q[..., :nb] = a * bits[perm]
    v = torch.randn(n, heads, t, d, generator=g)
    v = _round(v + torch.where(v < 0, -0.0625, 0.0625), dtype)
    expected = merge_heads(torch.gather(v, 2, perm[..., None].expand(-1, -1, -1, d)))
    return _pack(q, _round(k, dtype), v, dtype, device), expected.to(dtype).to(device), perm


def uniform_negative(n, t, heads, d, seed, dtype=torch.bfloat16, device="cpu"):
    """Every valid key scores -64 / sqrt(d) (-8 at d = 64) for every query, while a key the kernel reads past the
    end (zero-filled by TMA, or left at zero in shared memory) would score exactly 0 and outweigh each valid key by
    e^(64 / sqrt(d)).  q[.., 0] = 64, k[.., 0] = -1, q = 0 in the other channels, random k there.
    Returns (qkv, expected [N, T, C] float64 = the mean of v over the t keys)."""
    g = _gen(seed)
    q = torch.zeros(n, heads, t, d)
    q[..., 0] = 64.0
    k = torch.randn(n, heads, t, d, generator=g)
    k[..., 0] = -1.0
    v = _round(torch.randn(n, heads, t, d, generator=g), dtype)
    expected = merge_heads(v.double().mean(dim=2, keepdim=True).expand(-1, -1, t, -1))
    return _pack(q, _round(k, dtype), v, dtype, device), expected.to(device)


def uniform_negative_bound(qkv, expected, out_rel=U_BF16):
    """Tolerance of `uniform_negative`: out_rel |ref| + 2^-12 mean_j |v_j| (per image and channel).  Every p_j is
    exactly 1 in both kernels, so what remains is the fp32 sum of t values and the output rounding."""
    c = qkv.shape[-1] // 3
    mean_abs_v = qkv[..., 2 * c:].double().abs().mean(dim=1, keepdim=True)
    return out_rel * expected.abs() + 2.0 ** -12 * mean_abs_v


RAMP_KINDS = ("rising", "falling", "spike")


def ramp(n, t, heads, d, seed, kind, dtype=torch.bfloat16, device="cpu"):
    """Scores with a trend over the key index, for the online-softmax rescale.  Returns qkv.

    Channel 0 carries the trend, the others a random part of standard deviation 0.25 logits.  Per query row i a
    random slope rho_i in [12, 24] logits over the whole sequence:
      * "rising":  score ~ rho_i j / t -- the trend rises by >= 1.5 logits per 128-key tile at t <= 1024, so every
        new tile holds a larger maximum, alpha < 1 at every tile boundary, and the earlier tiles still carry weight;
      * "falling": score ~ rho_i (t - 1 - j) / t -- the maximum is in the first tile, alpha = 1 afterwards;
      * "spike":   random scores plus one key, at a random position in the last 128-key tile (partial unless
        t % 128 == 0), ln(t) + rho_i / 12 - 1.5 logits above zero: the maximum jumps at the last tile while the
        other keys keep between about a third and two thirds of the weight.
    """
    assert kind in RAMP_KINDS, kind
    g = _gen(seed)
    rho = 12.0 + 12.0 * torch.rand(n, heads, t, generator=g)
    rd = math.sqrt(d)
    q = torch.randn(n, heads, t, d, generator=g) * 0.25
    k = torch.randn(n, heads, t, d, generator=g)
    j = torch.arange(t, dtype=torch.float32)
    if kind == "spike":
        last0 = (t - 1) // 128 * 128
        spike = torch.randint(last0, t, (n, heads, 1, 1), generator=g)
        k[..., 0] = 0.0
        k.scatter_(2, spike.expand(-1, -1, 1, d), 0.0)
        k[..., 0].scatter_(2, spike[..., 0], 1.0)
        q[..., 0] = (math.log(t) + rho / 12.0 - 1.5) * rd
    else:
        trend = j / t if kind == "rising" else (t - 1 - j) / t
        k[..., 0] = 8.0 * trend
        q[..., 0] = rho * rd / 8.0
    v = torch.randn(n, heads, t, d, generator=g)
    return _pack(_round(q, dtype), _round(k, dtype), _round(v, dtype), dtype, device)
