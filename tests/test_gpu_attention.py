"""tcgen05 fused attention (forward + backward) vs an fp32 PyTorch reference of the same op."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu


def _api():
    from bert_pytorch_b200 import ops
    from bert_pytorch_b200.ops import api
    assert ops.available()
    return api


def _ref(qkv, seqlens, heads):
    B, S, H3 = qkv.shape
    H = H3 // 3
    d = H // heads
    t = qkv.float().view(B, S, 3, heads, d)
    q, k, v = (t[:, :, i].transpose(1, 2) for i in range(3))
    scores = q @ k.transpose(-1, -2) / math.sqrt(d)
    mask = torch.arange(S, device=qkv.device)[None, :] < seqlens[:, None]
    scores = scores.masked_fill(~mask[:, None, None, :], float("-inf"))
    p = torch.softmax(scores, dim=-1)
    lse = torch.logsumexp(scores, dim=-1)
    return (p @ v).transpose(1, 2).reshape(B, S, H), lse


def _ref_dropout(qkv, seqlens, heads, dctx, p_drop, seed, stream):
    """fp32 forward and backward of attention with the kernels' dropout on the probabilities: the keep mask is
    regenerated from the kernels' Philox counters (element ((b * heads + h) * S + q) * S + k, utils/philox.py).  Values
    are rounded to bf16 where the kernels round them:
      * P~ = P * keep / keep_prob, before P~ V (the context) and P~^T dO (dV); the forward kernels round P~ before
        dividing by the row sum, so there the rounding is mirrored only up to the scale;
      * the context, which the backward kernels read back for delta = <dO, O>;
      * dS = P * (dP * keep / keep_prob - delta) * scale, before dS^T Q (dK) and dS K (dQ).
    Returns the context [B, S, H], the log-sum-exp [B, heads, S] and dqkv [B, S, 3H], all fp32."""
    from bert_pytorch_b200.utils import philox
    B, S, H3 = qkv.shape
    H = H3 // 3
    d = H // heads
    t = qkv.float().view(B, S, 3, heads, d)
    q, k, v = (t[:, :, i].transpose(1, 2) for i in range(3))
    scale = 1.0 / math.sqrt(d)
    scores = (q @ k.transpose(-1, -2)) * scale
    mask = torch.arange(S, device=qkv.device)[None, :] < seqlens[:, None]
    scores = scores.masked_fill(~mask[:, None, None, :], float("-inf"))
    lse = torch.logsumexp(scores, dim=-1)
    p = torch.exp(scores - lse[..., None])
    keep = torch.from_numpy(philox.keep_mask(seed, stream, B * heads * S * S, p_drop)).to(qkv.device)
    drop = keep.view(B, heads, S, S).float() * philox.keep_scale(p_drop)
    pt = (p * drop).bfloat16().float()
    ctx = pt @ v
    do = dctx.float().view(B, S, heads, d).transpose(1, 2)
    delta = (do * ctx.bfloat16().float()).sum(-1, keepdim=True)
    ds = (p * ((do @ v.transpose(-1, -2)) * drop - delta) * scale).bfloat16().float()
    dqkv = torch.stack([ds @ k, ds.transpose(-1, -2) @ q, pt.transpose(-1, -2) @ do], dim=1)      # [B, 3, heads, S, d]
    return ctx.transpose(1, 2).reshape(B, S, H), lse, dqkv.permute(0, 3, 1, 2, 4).reshape(B, S, 3 * H)


@pytest.mark.parametrize("B,S,heads,lens", [
    (2, 128, 2, [128, 77]), (3, 128, 4, [128, 1, 64]), (2, 256, 2, [256, 130]), (2, 512, 2, [512, 300]),
    (2, 384, 2, [384, 129]), (1, 64, 2, [50]),
])
def test_attention_fwd_bwd_no_dropout(B, S, heads, lens):
    K = _api()
    torch.manual_seed(0)
    H = heads * 64
    qkv = (torch.randn(B, S, 3 * H, device="cuda") * 0.7).to(torch.bfloat16)
    seqlens = torch.tensor(lens, device="cuda", dtype=torch.int32)
    ctx, lse = K.attention_fwd(qkv, seqlens, heads)
    leaf = qkv.float().requires_grad_(True)
    ref, ref_lse = _ref(leaf, seqlens, heads)
    err = (ctx.float() - ref).abs().max().item()
    assert err < 2e-2, err
    assert (lse - ref_lse).abs().max().item() < 2e-2
    dctx = (torch.randn(B, S, H, device="cuda") * 0.5).to(torch.bfloat16)
    ref.backward(dctx.float())
    dqkv = K.attention_bwd(qkv, seqlens, ctx, dctx, lse, heads)
    g = leaf.grad
    scale = g.abs().max().item()
    # padded *keys* get exactly zero dK/dV in both; compare everything
    err = (dqkv.float() - g).abs().max().item()
    assert err < 4e-2 * max(scale, 1.0), (err, scale)


@pytest.mark.parametrize("S", [256, 128])          # 128: the single-block kernels (two / three CTAs per SM)
def test_attention_dropout_statistics_and_adjoint(S):
    K = _api()
    torch.manual_seed(0)
    B, heads = 2, 2
    H = heads * 64
    qkv = (torch.randn(B, S, 3 * H, device="cuda") * 0.5).to(torch.bfloat16)
    seqlens = torch.tensor([S, S - 56], device="cuda", dtype=torch.int32)
    base, _ = K.attention_fwd(qkv, seqlens, heads)
    outs = [K.attention_fwd(qkv, seqlens, heads, p_drop=0.1, seed=1000 + i, stream=3)[0].float() for i in range(24)]
    again = K.attention_fwd(qkv, seqlens, heads, p_drop=0.1, seed=1000, stream=3)[0].float()
    assert torch.equal(outs[0], again)                       # deterministic in (seed, stream)
    assert not torch.equal(outs[0], outs[1])
    mean = torch.stack(outs).mean(0)
    assert (mean - base.float()).abs().mean().item() < 2e-2   # unbiased
    # adjoint identity in V for a fixed mask: <dO, O(V)> == <dV, V>  (O is linear in V)
    ctx, lse = K.attention_fwd(qkv, seqlens, heads, p_drop=0.1, seed=7, stream=3)
    # dO correlated with O so that <dO, O> is a large positive number: a 1 / keep_prob slip between the forward and the
    # backward mask scaling (11 %) cannot hide behind cancellation
    dctx = (ctx.float() * 4.0 + 0.25 * torch.randn(B, S, H, device="cuda")).to(torch.bfloat16)
    dqkv = K.attention_bwd(qkv, seqlens, ctx, dctx, lse, heads, p_drop=0.1, seed=7, stream=3)
    lhs = (dctx.float() * ctx.float()).sum().item()
    v = qkv.float().view(B, S, 3, H)[:, :, 2]
    dv = dqkv.float().view(B, S, 3, H)[:, :, 2]
    rhs = (dv * v).sum().item()
    assert lhs > 50.0 and abs(lhs - rhs) < 2e-2 * abs(lhs), (lhs, rhs)
    # and with a different seed the identity must break (proves the mask really matters)
    dqkv2 = K.attention_bwd(qkv, seqlens, ctx, dctx, lse, heads, p_drop=0.1, seed=8, stream=3)
    rhs2 = (dqkv2.float().view(B, S, 3, H)[:, :, 2] * v).sum().item()
    assert abs(rhs2 - rhs) > 1e-3 * max(abs(rhs), 1.0)


@pytest.mark.parametrize("B,S,heads,lens,p_drop", [
    (3, 128, 4, [128, 77, 1], 0.1), (2, 128, 2, [128, 64], 0.0), (2, 64, 2, [64, 50], 0.1),
    (3, 512, 4, [512, 300, 129], 0.1), (2, 256, 2, [256, 130], 0.1), (2, 384, 2, [384, 1], 0.0), (40, 128, 16, None, 0.1),
    (2, 512, 2, [512, 300], 0.0), (2, 256, 2, [256, 130], 0.0), (2, 384, 2, [384, 129], 0.0), (3, 512, 4, [512, 1, 200], 0.1),
])
def test_attention_matches_fp32_dropout_oracle(B, S, heads, lens, p_drop):
    """Forward and backward kernels against ``_ref_dropout`` on the same inputs and the same dropout stream: context
    and log-sum-exp on the valid query rows, dQ/dK/dV everywhere.  S <= 128 runs attn_fwd_row_kernel and
    attn_bwd_row2_kernel, S > 128 attn_fwd_stream_kernel and attn_bwd_pipe_kernel; the 40 x 16 case has more items than
    resident CTAs (exercises the persistent loops)."""
    K = _api()
    torch.manual_seed(2)
    H = heads * 64
    qkv = (torch.randn(B, S, 3 * H, device="cuda") * 0.7).to(torch.bfloat16)
    seqlens = torch.tensor(lens if lens is not None else [S - (i % 5) * 7 for i in range(B)], device="cuda", dtype=torch.int32)
    dctx = (torch.randn(B, S, H, device="cuda") * 0.5).to(torch.bfloat16)
    kw = dict(p_drop=p_drop, seed=99, stream=6)
    ctx0, lse0, g0 = _ref_dropout(qkv, seqlens, heads, dctx, **kw)
    valid = torch.arange(S, device="cuda")[None, :] < seqlens[:, None]                  # padded query rows: don't care
    tol = 1.5e-2 * max(g0.abs().max().item(), 1.0)
    for _ in range(2):                                       # twice: races show up as run-to-run differences
        ctx, lse = K.attention_fwd(qkv, seqlens, heads, **kw)
        g = K.attention_bwd(qkv, seqlens, ctx, dctx, lse, heads, **kw).float()
        torch.cuda.synchronize()
        assert ((ctx.float() - ctx0).abs() * valid[:, :, None]).max().item() < 2e-2
        assert ((lse - lse0).abs() * valid[:, None, :]).max().item() < 1e-3
        assert (g - g0).abs().max().item() <= tol, ((g - g0).abs().max().item(), tol)
    if p_drop > 0.0:
        # the oracle fed the masks of another seed must miss by far: the comparison above really checks the masks
        _, _, g1 = _ref_dropout(qkv, seqlens, heads, dctx, p_drop=p_drop, seed=100, stream=6)
        assert (g - g1).abs().max().item() > 4 * tol, ((g - g1).abs().max().item(), tol)
