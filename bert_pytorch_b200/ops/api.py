"""Python wrappers over the sm_100a extension (``_C.so``).

Thin: allocate outputs, pick tile/split heuristics, translate enums.  No autograd here -- the
fused engine (models/fused.py) calls forward and backward kernels explicitly.
"""
from __future__ import annotations

import math
import os
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import extension

# GEMM enums (csrc/gemm_sm100.h)
NT, NN, TN = 0, 1, 2
(EPI_NONE, EPI_BIAS, EPI_BIAS_GELU, EPI_BIAS_DROP_RES, EPI_ADD, EPI_DGELU, EPI_ACCUM_F32, EPI_BIAS_TANH, EPI_F32,
 EPI_BIAS_GELU_DG, EPI_MUL) = range(11)

NUM_SMS = 148
_PAIR_ENABLED = os.environ.get("B200_GEMM_PAIR", "1") != "0"
KERNEL_LAUNCHES = 0     # every wrapper bumps this: bench.py reports it as ``gpu_launches``


# stream-K weight gradients: measured slower than 2-4 way split-K on the BERT-large shapes (operands of
# neighbouring clusters stop sharing L2 lines: profiles/gemm_bench_r1_v3_streamk.jsonl), so opt-in
STREAM_K = os.environ.get("B200_STREAM_K", "0") == "1"
# tail split (idle CTA pairs take the K tails): +3 % on the 48-tile QKV weight gradient, -8 % on the 64-tile FFN
# ones (each helper pays one fp32 red epilogue per tail piece) -> opt-in as well
TAIL_SPLIT = os.environ.get("B200_TAIL_SPLIT", "0") == "1"


def pick_block_n(M: int, N: int) -> int:
    """The tile variant :func:`gemm` chooses for an [M, N] output (512 = CTA-pair kernel)."""
    return _pick_block_n(M, N)


def _count(n: int = 1) -> None:
    global KERNEL_LAUNCHES
    KERNEL_LAUNCHES += n


def _pick_block_n(M: int, N: int) -> int:
    """512 = CTA-pair kernel (256 x 256 tile per 2-CTA cluster, tcgen05 cta_group::2): the default for the
    large GEMMs; 256 / 128 = single-CTA 128 x N tiles for small or skinny problems."""
    if M > 128 and N > 128 and _PAIR_ENABLED:
        return 512
    if N <= 128:
        return 128
    m_blocks = (M + 127) // 128
    t256 = m_blocks * ((N + 255) // 256)
    t128 = m_blocks * ((N + 127) // 128)

    def eff(tiles: int, width: int) -> float:
        waves = math.ceil(tiles / NUM_SMS)
        return tiles * width / (waves * NUM_SMS * width) if tiles else 0.0
    return 256 if eff(t256, 256) >= eff(t128, 128) - 0.08 else 128


def gemm(a: torch.Tensor, b: torch.Tensor, *, layout: int = NT, epi: int = EPI_NONE,
         out: Optional[torch.Tensor] = None, bias: Optional[torch.Tensor] = None,
         res: Optional[torch.Tensor] = None, aux_out: Optional[torch.Tensor] = None, k_splits: int = 1,
         block_n: Optional[int] = None, alpha: float = 1.0, p_drop: float = 0.0, seed: int = 0,
         stream: int = 0, scale_a: Optional[torch.Tensor] = None, scale_b: Optional[torch.Tensor] = None,
         a_e5m2: bool = False, b_e5m2: bool = False, push: bool = False,
         colsum: Optional[torch.Tensor] = None, mask_out: Optional[torch.Tensor] = None,
         mask_in: Optional[torch.Tensor] = None) -> torch.Tensor:
    """tcgen05 GEMM with a fused epilogue (see csrc/gemm_sm100.cu).  ``a``/``b`` are 2-D bf16, or -- with
    ``scale_a``/``scale_b`` (device inv-scale scalars from an :class:`Fp8Meta`) -- 1-byte fp8 tensors.
    ``colsum`` (fp32 [N], EPI_NONE / EPI_ADD / EPI_MUL): accumulates the column sums of the bf16 output (a bias
    gradient that would otherwise need its own pass over the tensor).  ``mask_out`` (uint8 [M, N / 8],
    EPI_BIAS_DROP_RES on the CTA-pair kernel): receives the dropout keep bits, which :func:`layer_norm_bwd` can read
    back (``keep_mask``) instead of regenerating them."""
    if layout == NT:
        M, N = a.size(0), b.size(0)
    elif layout == NN:
        M, N = a.size(0), b.size(1)
    else:
        M, N = a.size(1), b.size(1)
    if out is None:
        dt = torch.float32 if epi in (EPI_ACCUM_F32, EPI_F32) else torch.bfloat16
        out = torch.empty(M, N, dtype=dt, device=a.device)
    if scale_a is not None:
        block_n = 512                      # fp8 operands run on the CTA-pair kernel
    elif block_n is None:
        block_n = _pick_block_n(M, N)
    extension().gemm(a, b, out, layout, epi, bias, res, aux_out, k_splits, block_n, alpha, p_drop, seed, stream,
                     scale_a, scale_b, a_e5m2, b_e5m2, push, colsum, mask_out, mask_in)
    _count()
    return out


def mx_quantize(x: torch.Tensor):
    """bf16 [R, K] -> (e4m3 bytes [R, K], ue8m0 block scales in the tensor-core layout): OCP MXFP8, one scale per
    32 elements along K (csrc/gemm_mx.cu)."""
    R, Kd = x.shape
    q = torch.empty(R, Kd, dtype=torch.uint8, device=x.device)
    sf = torch.empty(((R + 127) // 128) * (Kd // 128) * 512, dtype=torch.uint8, device=x.device)
    extension().mx_quantize(x, q, sf)
    _count()
    return q, sf


def mx_dequantize(q: torch.Tensor, sf: torch.Tensor) -> torch.Tensor:
    """fp32 view of an MXFP8 tensor (test / debugging aid; plain torch)."""
    R, Kd = q.shape
    rows = torch.arange(R, device=q.device)
    groups = torch.arange(Kd // 32, device=q.device)
    idx = ((rows[:, None] // 128) * (Kd // 128) + groups[None, :] // 4) * 512 + (rows[:, None] % 32) * 16 \
        + ((rows[:, None] // 32) % 4) * 4 + groups[None, :] % 4
    scale = torch.exp2(sf.long()[idx].float() - 127.0)                    # [R, K/32]
    return q.view(torch.float8_e4m3fn).float() * scale.repeat_interleave(32, dim=1)


def gemm_mx(a_q: torch.Tensor, a_sf: torch.Tensor, b_q: torch.Tensor, b_sf: torch.Tensor, *,
            bias: Optional[torch.Tensor] = None, out_dtype: torch.dtype = torch.bfloat16) -> torch.Tensor:
    """D = A . B^T on block-scaled fp8 operands (tcgen05.mma.kind::mxf8f6f4.block_scale, scales staged in TMEM)."""
    out = torch.empty(a_q.size(0), b_q.size(0), dtype=out_dtype, device=a_q.device)
    extension().gemm_mxfp8(a_q, a_sf, b_q, b_sf, out, bias)
    _count()
    return out


class Fp8Meta:
    """Device-resident per-tensor scaling records ``{amax, scale, inv_scale, _}`` for the fp8 GEMM path
    (delayed scaling: quantise with the scale derived from the previous step's amax; csrc/fp8.cu)."""

    def __init__(self, sites: Sequence[str], e5m2: Sequence[bool], device, margin: float = 1.0):
        self.index = {name: i for i, name in enumerate(sites)}
        self.e5m2 = list(bool(x) for x in e5m2)
        self.table = torch.zeros(len(sites), 4, dtype=torch.float32, device=device)
        self.table[:, 1:3] = 1.0
        self.flags = torch.tensor([1 if x else 0 for x in self.e5m2], dtype=torch.int32, device=device)
        self.margin = float(margin)

    def record(self, site) -> torch.Tensor:
        return self.table[self.index[site] if isinstance(site, str) else site]

    def inv_scale(self, site) -> torch.Tensor:
        return self.record(site)[2:3]

    def is_e5m2(self, site) -> bool:
        return self.e5m2[self.index[site] if isinstance(site, str) else site]

    def quantize(self, x: torch.Tensor, site, out: Optional[torch.Tensor] = None, calibrate: bool = False) -> torch.Tensor:
        """bf16 -> fp8 bytes with the site's current scale; records amax for the next ``update``.  With
        ``calibrate`` the scale is first derived from this very tensor (current scaling, one extra pass)."""
        ext = extension()
        rec = self.record(site)
        e5 = self.is_e5m2(site)
        if calibrate:
            ext.fp8_amax(x, rec)
            i = self.index[site] if isinstance(site, str) else site
            ext.fp8_update(self.table[i:i + 1], self.flags[i:i + 1], self.margin)
            _count(2)
        if out is None:
            out = torch.empty(x.shape, dtype=torch.uint8, device=x.device)
        ext.fp8_quantize(x, out, rec, e5)
        _count()
        return out

    def update(self) -> None:
        """new scales from the amaxes seen since the last update (one tiny launch for all sites)"""
        extension().fp8_update(self.table, self.flags, self.margin)
        _count()


# opt-in: 256 x 512 weight-gradient tiles measured faster in isolation (0.088 vs 0.096 ms, FFN shapes) but slower inside
# the training step (74.5 vs 62.9 us per call, side stream off) -- profiles/README.md
WGRAD_WIDE = os.environ.get("B200_WGRAD_WIDE", "0") == "1"


def wgrad_splits(n_out: int, k_out: int, reduce_len: int, block_n: int = 256) -> int:
    """Split-K factor for dW[n_out, k_out] so the grid covers the machine."""
    if block_n == 512:
        tiles = ((n_out + 255) // 256) * ((k_out + 255) // 256)
        units = NUM_SMS // 2
    else:
        tiles = ((n_out + 127) // 128) * ((k_out + block_n - 1) // block_n)
        units = NUM_SMS
    kb = max(1, (reduce_len + 63) // 64)
    want = max(1, round(2 * units / max(tiles, 1)))
    return max(1, min(want, kb // 4 if kb >= 8 else 1, 32))


def wgrad_accumulate(dy: torch.Tensor, x: torch.Tensor, grad: torch.Tensor, alpha: float = 1.0, push: bool = False,
                     **fp8) -> None:
    """grad[N,K] (fp32, arena view) += dy[M,N]^T @ x[M,K]  (``fp8``: scale_a / scale_b / a_e5m2 for 1-byte operands)."""
    n_out, k_out = grad.shape
    bn = 512 if fp8 else _pick_block_n(n_out, k_out)
    if bn == 128 and k_out >= 256:
        bn = 256
    if bn == 512 and not fp8 and WGRAD_WIDE and k_out % 512 == 0:
        # 256 x 512 tiles (two N = 256 MMAs per k-step share the A operand: a quarter fewer operand bytes per FLOP, which
        # is what the MN-major TMA supply of the TN kernel is short of); fewer tiles than CTA pairs -> tail split
        tiles = ((n_out + 255) // 256) * (k_out // 512)
        kb = (dy.size(0) + 63) // 64
        pairs = NUM_SMS // 2
        splits = -2 if (tiles < pairs and kb * tiles // pairs >= 4) else 1
        gemm(dy, x, layout=TN, epi=EPI_ACCUM_F32, out=grad, block_n=1024, alpha=alpha, k_splits=splits, push=push)
        return
    splits = wgrad_splits(n_out, k_out, dy.size(0) // (2 if fp8 else 1), bn)
    if bn == 512 and not fp8 and not TAIL_SPLIT and not STREAM_K:
        # round-2 measurement with the 7-stage operand ring (profiles/gemm_bench_r2_wgrad.jsonl): the 48-tile QKV
        # weight gradient gains 6 % from the tail split (1179 vs 1110 TFLOP/s), the 64-tile FFN ones lose 18 %
        tiles = ((n_out + 255) // 256) * ((k_out + 255) // 256)
        if 40 <= tiles <= 56:
            splits = -2
    if bn == 512 and TAIL_SPLIT:
        # fewer tiles than CTA pairs and a split-K grid that leaves > 7 % of the machine idle in its last wave:
        # tail split (cluster t runs the head of tile t's K range, the idle clusters share the tails; gemm_sm100.cu)
        tiles = ((n_out + 255) // 256) * ((k_out + 255) // 256)
        pairs = NUM_SMS // 2
        kb = (dy.size(0) + (127 if fp8 else 63)) // (128 if fp8 else 64)
        if tiles < pairs:
            units = tiles * max(splits, 1)
            eff = units / (((units + pairs - 1) // pairs) * pairs)
            if eff < 0.93 and kb * tiles // pairs >= 4:
                splits = -2
    if bn == 512 and STREAM_K:
        # stream-K: equal (tile, k-block) ranges per CTA pair instead of whole tiles (csrc/gemm_sm100.cu: seg_get)
        tiles = ((n_out + 255) // 256) * ((k_out + 255) // 256)
        kb = (dy.size(0) + (127 if fp8 else 63)) // (128 if fp8 else 64)
        if tiles % (NUM_SMS // 2) != 0 and tiles * kb >= 8 * (NUM_SMS // 2):
            splits = -1
    # ``push``: with the peer-memory backend in push mode the tiles go to the owner rank's arena (GEMM -> reduce-scatter)
    gemm(dy, x, layout=TN, epi=EPI_ACCUM_F32, out=grad, block_n=bn, alpha=alpha, k_splits=splits, push=push, **fp8)


def _fp8_side(fp8, like: torch.Tensor):
    """``fp8`` = (Fp8Meta, site) -> (q tensor, meta record, e5m2) for a kernel's fused fp8 copy of its output."""
    if fp8 is None:
        return None, None, False
    meta, site = fp8
    return torch.empty(like.shape, dtype=torch.uint8, device=like.device), meta.record(site), meta.is_e5m2(site)


def layer_norm_fwd(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, *, eps: float = 1e-12,
                   save_stats: bool = True, p_drop: float = 0.0, seed: int = 0, stream: int = 0, fp8=None):
    """``fp8=(meta, site)``: also emit the fp8 copy of y (delayed scaling) -> returns (y, mean, rstd, q)."""
    y = torch.empty_like(x)
    M = x.numel() // x.size(-1)
    mean = torch.empty(M, dtype=torch.float32, device=x.device) if save_stats else None
    rstd = torch.empty(M, dtype=torch.float32, device=x.device) if save_stats else None
    q, rec, e5 = _fp8_side(fp8, x)
    extension().layer_norm_fwd(x, gamma, beta, y, mean, rstd, eps, p_drop, seed, stream, q, rec, e5)
    _count()
    return (y, mean, rstd) if fp8 is None else (y, mean, rstd, q)


_LN_WS: Dict[Tuple[int, int, int], torch.Tensor] = {}


def _ln_workspace(M: int, H: int, device: torch.device) -> torch.Tensor:
    key = (device.index or 0, M, H)
    ws = _LN_WS.get(key)
    if ws is None:
        ws = torch.empty(extension().ln_bwd_workspace(M, H), dtype=torch.float32, device=device)
        _LN_WS[key] = ws
    return ws


NO_STREAM = 0xFFFFFFFF


def dropout_mask(M: int, N: int, p_drop: float, seed: int, stream: int, device) -> torch.Tensor:
    """uint8 [M, N / 8] keep bits of the dropout stream ``(seed, stream)`` over an [M, N] tensor -- the decisions the
    kernels would draw themselves.  Feed it to ``gemm(..., mask_in=)`` (EPI_BIAS_DROP_RES) and to
    ``layer_norm_bwd(..., keep_mask=)``: Philox then runs once per element, in a kernel that keeps the whole machine
    busy, instead of in the latency-bound GEMM epilogue and again in the LayerNorm backward."""
    out = torch.empty(M, N // 8, dtype=torch.uint8, device=device)
    extension().dropout_mask(out, p_drop, seed, stream)
    _count()
    return out


def layer_norm_bwd(dy: torch.Tensor, x: torch.Tensor, mean: torch.Tensor, rstd: torch.Tensor, gamma: torch.Tensor, *,
                   dgamma: Optional[torch.Tensor], dbeta: Optional[torch.Tensor], dbias: Optional[torch.Tensor] = None,
                   want_dropped: bool = False, p_drop: float = 0.0, seed: int = 0, drop_stream: int = 0,
                   in_stream: int = NO_STREAM, fp8=None, keep_mask: Optional[torch.Tensor] = None):
    """Returns (dx, dx_dropped or None).  ``dgamma``/``dbeta``/``dbias`` are *accumulated into*.
    ``keep_mask`` (uint8 [M, H / 8]): the keep bits of the ``drop_stream`` dropout as written by the producing GEMM
    (``gemm(mask_out=...)``); without it the decisions are regenerated from the Philox stream (same bits).
    ``fp8=(meta, site)`` (with ``want_dropped``): also the fp8 copy of dx_dropped -> (dx, dxd, q)."""
    dx = torch.empty_like(x)
    dxd = torch.empty_like(x) if want_dropped else None
    M, H = x.numel() // x.size(-1), x.size(-1)
    q, rec, e5 = _fp8_side(fp8 if want_dropped else None, x)
    extension().layer_norm_bwd(dy, x, mean, rstd, gamma, dx, dxd, dgamma, dbeta, dbias, _ln_workspace(M, H, x.device),
                               p_drop, seed, drop_stream, in_stream, q, rec, e5, keep_mask)
    _count(2)
    return (dx, dxd) if fp8 is None else (dx, dxd, q)


def colsum_accumulate(x: torch.Tensor, out: torch.Tensor) -> None:
    """out[N] (fp32) += x[M,N].sum(0)"""
    extension().colsum(x, out)
    _count()


def gelu_fwd(x: torch.Tensor, fp8=None):
    y = torch.empty_like(x)
    q, rec, e5 = _fp8_side(fp8, x)
    extension().gelu_fwd(x, y, q, rec, e5)
    _count()
    return y if fp8 is None else (y, q)


def dgelu_bwd(dy: torch.Tensor, x: torch.Tensor, dbias: Optional[torch.Tensor] = None, fp8=None):
    """dy * gelu'(x); ``dbias`` (fp32 [N]) accumulates the column sums of the result."""
    dx = torch.empty_like(dy)
    q, rec, e5 = _fp8_side(fp8, dy)
    extension().dgelu_bwd(dy, x, dx, dbias, q, rec, e5)
    _count()
    return dx if fp8 is None else (dx, q)


def embedding_fwd(ids, seg, word, pos, type_emb, gamma, beta, S: int, *, eps=1e-12, p_drop=0.0, seed=0, stream=0):
    M, H = ids.numel(), word.size(1)
    e = torch.empty(M, H, dtype=torch.bfloat16, device=ids.device)
    y = torch.empty_like(e)
    mean = torch.empty(M, dtype=torch.float32, device=ids.device)
    rstd = torch.empty_like(mean)
    extension().embedding_fwd(ids, seg, word, pos, type_emb, gamma, beta, e, y, mean, rstd, S, eps, p_drop, seed, stream)
    _count()
    return y, e, mean, rstd


def embedding_bwd_scatter(de, ids, seg, gword, gpos, gtype, S: int) -> None:
    extension().embedding_bwd_scatter(de, ids, seg, gword, gpos, gtype, S)
    _count()


def mlm_compact(labels: torch.Tensor, max_pred: int):
    B = labels.size(0)
    idx = torch.empty(B * max_pred, dtype=torch.int32, device=labels.device)
    tgt = torch.empty_like(idx)
    count = torch.empty(1, dtype=torch.int32, device=labels.device)
    extension().mlm_compact(labels, max_pred, idx, tgt, count)
    _count()
    return idx, tgt, count


def gather_rows(src: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
    dst = torch.empty(idx.numel(), src.size(-1), dtype=src.dtype, device=src.device)
    extension().gather_rows(src, idx, dst)
    _count()
    return dst


def scatter_rows(src: torch.Tensor, idx: torch.Tensor, dst: torch.Tensor) -> None:
    extension().scatter_rows(src, idx, dst)
    _count()


def nsp_head_(pooled: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, labels: torch.Tensor, grad_scale: float,
              loss_out: torch.Tensor, dw: torch.Tensor, db: torch.Tensor) -> torch.Tensor:
    """NSP classifier [B,H] x [H,2] + cross-entropy (ignore_index -1) + backward in one launch: ``loss_out`` += mean CE,
    ``dw`` / ``db`` (fp32) accumulate the classifier gradients, returns dz = d loss / d (pooler pre-activation) [B,H]
    bf16 (tanh' of the pooler folded in)."""
    dz = torch.empty_like(pooled)
    extension().nsp_head(pooled, w, bias, labels, grad_scale, loss_out, dz, dw, db)
    _count()
    return dz


def softmax_ce_(logits: torch.Tensor, targets: torch.Tensor, count: torch.Tensor, grad_scale: float,
                loss_out: torch.Tensor) -> None:
    """In place: logits <- d loss / d logits (scaled); loss_out += mean CE over valid targets."""
    extension().softmax_ce(logits, targets, count, grad_scale, loss_out)
    _count()


def attention_fwd(qkv: torch.Tensor, seqlens: torch.Tensor, heads: int, *, p_drop=0.0, seed=0, stream=0, fp8=None):
    """``fp8=(meta, site)``: the kernel also writes the fp8 copy of the context -> (ctx, lse, q)."""
    B, S, H3 = qkv.shape
    H = H3 // 3
    ctx = torch.empty(B, S, H, dtype=torch.bfloat16, device=qkv.device)
    lse = torch.empty(B, heads, S, dtype=torch.float32, device=qkv.device)
    q, rec, e5 = _fp8_side(fp8, ctx)
    extension().attention_fwd(qkv, seqlens, ctx, lse, heads, 1.0 / math.sqrt(H // heads), p_drop, seed, stream, q, rec, e5)
    _count()
    return (ctx, lse) if fp8 is None else (ctx, lse, q)


def attention_bwd(qkv, seqlens, ctx, dctx, lse, heads: int, *, p_drop=0.0, seed=0, stream=0, fp8=None):
    """``fp8=(meta, site)``: the kernels also write the fp8 copy of dqkv -> (dqkv, q)."""
    B, S, H3 = qkv.shape
    H = H3 // 3
    dqkv = torch.empty_like(qkv)
    delta = torch.empty(B, heads, S, dtype=torch.float32, device=qkv.device)
    dq_acc = torch.empty(B * S, H, dtype=torch.float32, device=qkv.device) if S > 128 else None
    q, rec, e5 = _fp8_side(fp8, dqkv)
    extension().attention_bwd(qkv, seqlens, ctx, dctx, lse, dqkv, delta, dq_acc, heads, 1.0 / math.sqrt(H // heads), p_drop,
                              seed, stream, q, rec, e5)
    _count(2)
    return dqkv if fp8 is None else (dqkv, q)


# ---------------------------------------------------------------------------
# multi-tensor ops over arbitrary tensor lists
# ---------------------------------------------------------------------------
CHUNK = 65536
_DT = {torch.float32: 0, torch.bfloat16: 1, torch.float16: 2}
_TABLE_CACHE: Dict[Tuple, Tuple[torch.Tensor, ...]] = {}


def _chunk_table(numels: Sequence[int], device: torch.device, offsets: Optional[Sequence[int]] = None):
    """chunk -> (tensor, start, len).  With ``offsets`` the starts are absolute arena positions."""
    ct, cs, cl = [], [], []
    for t, n in enumerate(numels):
        base = offsets[t] if offsets is not None else 0
        for s in range(0, n, CHUNK):
            ct.append(t); cs.append(base + s); cl.append(min(CHUNK, n - s))
    return (torch.tensor(ct, dtype=torch.int32, device=device), torch.tensor(cs, dtype=torch.int64, device=device),
            torch.tensor(cl, dtype=torch.int32, device=device))


def _list_tables(tensors: List[torch.Tensor]):
    key = tuple((t.data_ptr(), t.numel()) for t in tensors)
    hit = _TABLE_CACHE.get(key)
    if hit is None:
        dev = tensors[0].device
        ptrs = torch.tensor([t.data_ptr() for t in tensors], dtype=torch.int64, device=dev)
        hit = (ptrs,) + _chunk_table([t.numel() for t in tensors], dev)
        if len(_TABLE_CACHE) > 64:
            _TABLE_CACHE.clear()
        _TABLE_CACHE[key] = hit
    return hit


def multi_tensor_l2norm(tensors: List[torch.Tensor], per_tensor: bool = False):
    dev = tensors[0].device
    total = torch.zeros(1, dtype=torch.float32, device=dev)
    per = torch.zeros(len(tensors), dtype=torch.float32, device=dev) if per_tensor else None
    by_dtype: Dict[torch.dtype, List[int]] = {}
    for i, t in enumerate(tensors):
        if not t.is_contiguous():
            raise ValueError("multi_tensor_l2norm needs contiguous tensors")
        by_dtype.setdefault(t.dtype, []).append(i)
    for dt, idxs in by_dtype.items():
        group = [tensors[i] for i in idxs]
        ptrs, ct, cs, cl = _list_tables(group)
        sub = torch.zeros(len(group), dtype=torch.float32, device=dev) if per_tensor else None
        extension().mt_l2norm(_DT[dt], ptrs, ct, cs, cl, sub, total)
        _count()
        if per_tensor:
            per[torch.tensor(idxs, device=dev)] = sub
    return total.sqrt().squeeze(0), (per.sqrt() if per_tensor else torch.zeros(0, device=dev))


def multi_tensor_scale(src: List[torch.Tensor], dst: List[torch.Tensor], scale) -> torch.Tensor:
    dev = src[0].device
    overflow = torch.zeros(1, dtype=torch.int32, device=dev)
    groups: Dict[Tuple[torch.dtype, torch.dtype], List[int]] = {}
    for i, (s, d) in enumerate(zip(src, dst)):
        groups.setdefault((s.dtype, d.dtype), []).append(i)
    sd = scale.to(device=dev, dtype=torch.float32).reshape(1) if torch.is_tensor(scale) else None
    sh = 1.0 if torch.is_tensor(scale) else float(scale)
    for (sdt, ddt), idxs in groups.items():
        ins, outs = [src[i] for i in idxs], [dst[i] for i in idxs]
        ip, ct, cs, cl = _list_tables(ins)
        op = _list_tables(outs)[0]
        extension().mt_scale(_DT[sdt], _DT[ddt], ip, op, ct, cs, cl, sd, sh, overflow)
        _count()
    return overflow.squeeze(0)


# ---------------------------------------------------------------------------
# arena optimizers
# ---------------------------------------------------------------------------

def _arena_tables(arena):
    t = getattr(arena, "_opt_tables", None)
    if t is None:
        dev = arena.device
        ct, cs, cl = _chunk_table([s.numel for s in arena.slots], dev, [s.offset for s in arena.slots])
        t = dict(ct=ct, cs=cs, cl=cl,
                 decay=torch.tensor([1 if s.decay else 0 for s in arena.slots], dtype=torch.int32, device=dev),
                 stats=torch.zeros(1, dtype=torch.float32, device=dev),
                 norms=torch.zeros(2 * len(arena.slots), dtype=torch.float32, device=dev))
        arena._opt_tables = t
    return t


def flat_unscale_(flat_grad: torch.Tensor, inv_scale: torch.Tensor, found_inf: torch.Tensor) -> None:
    extension().flat_unscale(flat_grad, inv_scale.reshape(1), found_inf.reshape(1))
    _count()


def _uniform(optimizer, key):
    vals = {repr(g[key]) for g in optimizer.param_groups}
    if len(vals) != 1:
        raise NotImplementedError(f"fused arena optimizer needs the same '{key}' in every param group")
    return optimizer.param_groups[0][key]


def arena_lamb_step(arena, optimizer, inv_scale=None, found_inf=None) -> None:
    """One LAMB step over the arena (3 launches + 2 memsets).  Weight decay is per slot (decay flag x
    the single non-zero group value), every other hyper-parameter must agree across groups -- which is
    how every runner builds its groups (run_pretraining.py:279-296)."""
    T = _arena_tables(arena)
    lr = _uniform(optimizer, "lr")
    b1, b2 = _uniform(optimizer, "betas")
    eps = _uniform(optimizer, "eps")
    wds = sorted({float(g["weight_decay"]) for g in optimizer.param_groups})
    wd = max(wds)
    for g in optimizer.param_groups:      # decay flag of a slot must agree with its group's decay
        pass
    step = int(optimizer.param_groups[0].get("step", 0)) + 1
    ext = extension()
    inv = inv_scale.reshape(1) if inv_scale is not None else None
    fi = found_inf.reshape(1) if found_inf is not None else None
    ext.flat_sumsq(arena.flat_grad, inv, T["stats"], fi)
    ext.arena_lamb(arena.flat_grad, arena.flat_param, arena.exp_avg, arena.exp_avg_sq, arena.flat_shadow, T["ct"],
                   T["cs"], T["cl"], T["decay"], T["stats"], T["norms"], inv, fi, float(lr), float(b1), float(b2),
                   float(eps), float(wd), step, bool(_uniform(optimizer, "bias_correction")),
                   bool(_uniform(optimizer, "grad_averaging")), float(_uniform(optimizer, "max_grad_norm") or 0.0),
                   bool(optimizer.adam_w_mode), bool(optimizer.use_nvlamb))
    _count(3)
    # apex semantics: the step counter only advances when the update was applied.  Keeping that exact
    # would need a host sync on found_inf; with a scaler we advance optimistically only when no scaler
    # is in play, otherwise we read the flag (fp16 path only -- bf16 never has a scaler).
    if fi is None or float(fi) == 0.0:
        for g in optimizer.param_groups:
            g["step"] = step
    optimizer.last_grad_norm = T["stats"].sqrt()


def arena_adam_step(arena, optimizer, inv_scale=None, found_inf=None) -> None:
    T = _arena_tables(arena)
    lr = _uniform(optimizer, "lr")
    b1, b2 = _uniform(optimizer, "betas")
    eps = _uniform(optimizer, "eps")
    wd = max(float(g["weight_decay"]) for g in optimizer.param_groups)
    step = int(optimizer.param_groups[0].get("step", 0)) + 1
    inv = inv_scale.reshape(1) if inv_scale is not None else None
    fi = found_inf.reshape(1) if found_inf is not None else None
    extension().arena_adam(arena.flat_grad, arena.flat_param, arena.exp_avg, arena.exp_avg_sq, arena.flat_shadow,
                           T["ct"], T["cs"], T["cl"], T["decay"], inv, fi, float(lr), float(b1), float(b2), float(eps),
                           float(wd), step, bool(_uniform(optimizer, "bias_correction")), bool(optimizer.adam_w_mode))
    _count()
    if fi is None or float(fi) == 0.0:
        for g in optimizer.param_groups:
            g["step"] = step
