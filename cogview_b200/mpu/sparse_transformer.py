"""Transformer stack — mirror of the reference's mpu/sparse_transformer.py: same class names, constructor
signatures, parameter names (state_dict keys) and forward signatures, computed by the sm_100a kernels.

  LayerNorm                     :40-44    abs-max pre-scaled LN            -> cv_layernorm_absmax_*
  GPT2ParallelSelfAttention     :46-169   QKV GEMM, attention, out-proj    -> cv_gemm_bf16, cv_attn_*
  GPT2ParallelMLP               :189-234  h->4h (+GELU), 4h->h             -> cv_gemm_bf16 (fused epilogues)
  GPT2ParallelTransformerLayer  :237-342  Sandwich-LN block                -> one fused autograd Function
  GPT2ParallelTransformer       :361-626  embeddings, masks, layer loop, mems

Data layout on the device: the residual stream is fp32 [b*s, h]; everything that feeds a GEMM is bf16;
Q/K/V stay packed as the QKV GEMM output [b, s, 3h] and are read in place by the attention kernel through
strided TMA tensor maps (no split / permute / contiguous copies); the attention context is written
token-major [b, s, h].  Each tensor's max|x| (needed by the next LayerNorm) is produced by the kernel
that writes it.
"""
import math
import os
import random

import weakref

import torch

from .. import ops
from .layers import ColumnParallelLinear, RowParallelLinear, _as_bf16
from .random import checkpoint, get_cuda_rng_tracker, next_dropout_site  # noqa: F401
from .utils import divide

LN_EPS_DEFAULT = 1.0e-5


# ----------------------------------------------------------------------------------------------------
# LayerNorm
# ----------------------------------------------------------------------------------------------------
class _LayerNormFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, eps):
        shape = x.shape
        x2 = x.reshape(-1, shape[-1])
        if x2.dtype not in (torch.float32, torch.bfloat16):
            x2 = x2.float()
        x2 = x2.contiguous()
        am = ops.absmax(x2)
        y, mean, rstd = ops.layernorm_absmax_fwd(x2, am, _as_bf16(weight), _as_bf16(bias), eps,
                                                 out_dtype=x2.dtype, save_stats=True)
        ctx.save_for_backward(x2, mean, rstd, _as_bf16(weight))
        ctx.meta = (shape, x.dtype, weight.dtype, bias.dtype)
        return y.view(shape).to(x.dtype)

    @staticmethod
    def backward(ctx, dy):
        x2, mean, rstd, w = ctx.saved_tensors
        shape, xdt, wdt, bdt = ctx.meta
        dy2 = dy.reshape(x2.shape).to(x2.dtype).contiguous()
        dx, dg, db = ops.layernorm_absmax_bwd(x2, dy2, mean, rstd, w, dx_dtype=x2.dtype)
        return dx.view(shape).to(xdt), dg.to(wdt), db.to(bdt), None


class LayerNorm(torch.nn.Module):
    """LayerNorm(x / (max|x| / 8)) — mpu/sparse_transformer.py:40-44 (the max is global and detached)."""

    def __init__(self, normalized_shape, eps=LN_EPS_DEFAULT, elementwise_affine=True):
        super().__init__()
        if isinstance(normalized_shape, int):
            normalized_shape = (normalized_shape,)
        assert len(normalized_shape) == 1 and elementwise_affine
        self.normalized_shape = tuple(normalized_shape)
        self.eps = eps
        self.elementwise_affine = True
        self.weight = torch.nn.Parameter(torch.ones(*normalized_shape))
        self.bias = torch.nn.Parameter(torch.zeros(*normalized_shape))

    def forward(self, x):
        return _LayerNormFn.apply(x, self.weight, self.bias, self.eps)


# ----------------------------------------------------------------------------------------------------
# functional attention entry points (same names as the reference's module-level functions)
# ----------------------------------------------------------------------------------------------------
_mask_cache = {}


def mask_to_sep(attention_mask, sq, sk):
    """Recognise the two mask families the reference builds ([1,1,sq,sk] lower-triangular, or the int-`sep`
    form of :477-489) and return `sep`; any other mask tensor is rejected (no kernel for arbitrary masks)."""
    if isinstance(attention_mask, int):
        return attention_mask
    if attention_mask.numel() == 1:
        return int(attention_mask.item())
    # The check below reads the mask back (one sync); cache the verdict per live tensor object.  The entry holds a
    # weak reference: a new tensor that happens to reuse a freed mask's address must not inherit its verdict.
    key = (attention_mask.data_ptr(), tuple(attention_mask.shape), attention_mask._version, sq, sk)
    hit = _mask_cache.get(key)
    if hit is not None and hit[0]() is attention_mask:
        return hit[1]
    m = attention_mask.reshape(-1, attention_mask.shape[-2], attention_mask.shape[-1])
    if m.shape[0] != 1 or m.shape[1] != sq or m.shape[2] != sk:
        raise ValueError('attention_mask must be [1, 1, %d, %d] or an int sep; got %s' % (sq, sk,
                                                                                         tuple(attention_mask.shape)))
    m = m[0].float()
    sep = int(m[0].sum().item()) - (sk - sq)
    sep = max(0, min(sep, sq))
    cols = torch.arange(sk, device=m.device).unsqueeze(0)
    rows = torch.arange(sq, device=m.device).unsqueeze(1)
    expect = ((cols < sep + (sk - sq)) | (cols <= rows + (sk - sq))).float()
    if not torch.equal(m, expect):
        raise NotImplementedError('only lower-triangular / int-sep attention masks are supported by the fused '
                                  'attention kernel (mpu/sparse_transformer.py:477-489 families)')
    if sep <= 1:
        sep = 0
    if len(_mask_cache) > 64:
        _mask_cache.clear()
    _mask_cache[key] = (weakref.ref(attention_mask), sep)
    return sep


def standard_attention(query_layer, key_layer, value_layer, attention_mask, attention_dropout=None):
    """mpu/sparse_transformer.py:652-673 on [b, np, s, hn] tensors (API parity; the fused layer path never
    materialises this layout).  Forward only (no autograd through this entry point).  An `attention_dropout` module in
    training mode applies its p inside the kernel (counter-based keep mask, seed drawn from torch's generator — the
    reference draws from the model-parallel RNG tracker, :665-667; masks are not bit-identical to torch's)."""
    b, nh, sq, hn = query_layer.shape
    sk = key_layer.shape[2]
    sep = mask_to_sep(attention_mask, sq, sk)

    def tok_major(t):
        return _as_bf16(t).permute(0, 2, 1, 3).reshape(b, t.shape[2], nh * hn).contiguous()

    drop = None
    if attention_dropout is not None and attention_dropout.training and attention_dropout.p > 0:
        drop = (float(attention_dropout.p), int(torch.randint(0, 2 ** 62, (1,)).item()), 0)
    res = ops.attn_fwd(tok_major(query_layer), tok_major(key_layer), tok_major(value_layer), nh, sep=sep, dropout=drop)
    ctx = res[0] if drop is not None else res
    return ctx.view(b, sq, nh, hn).permute(0, 2, 1, 3).to(query_layer.dtype)


# ----------------------------------------------------------------------------------------------------
# fused transformer layer
# ----------------------------------------------------------------------------------------------------
_PARAM_ORDER = ('input_layernorm.weight', 'input_layernorm.bias',
                'attention.query_key_value.weight', 'attention.query_key_value.bias',
                'attention.dense.weight', 'attention.dense.bias',
                'third_layernorm.weight', 'third_layernorm.bias',
                'post_attention_layernorm.weight', 'post_attention_layernorm.bias',
                'mlp.dense_h_to_4h.weight', 'mlp.dense_h_to_4h.bias',
                'mlp.dense_4h_to_h.weight', 'mlp.dense_4h_to_h.bias',
                'fourth_layernorm.weight', 'fourth_layernorm.bias')


class SparseSpec:
    """Attention pattern of sparse TRAINING (is_sparse == 1, mpu/sparse_transformer.py:675-725): takes the place of
    the int `sep` in layer_forward / layer_backward.  pivot_idx: int64 [b, n_piv] on the device."""

    def __init__(self, pivot_idx, query_window, key_window_times):
        self.pivot_idx = pivot_idx.contiguous()
        self.w = int(query_window)
        self.times = int(key_window_times)


def layer_forward(x, am_x, P, heads, eps, b, sq, sep, kv=None, save=None, attn=None, drops=None):
    """One Sandwich-LN block (mpu/sparse_transformer.py:314-342) on the fp32 residual stream x [b*sq, h].

    am_x: 1-element fp32 tensor holding max|x|.  P: the 16 parameters in _PARAM_ORDER (bf16).
    kv: None (keys/values are this call's tokens) or a callable (k_new, v_new) -> (k_all, v_all) views used by
        the KV-cache path.  save: None or a list that receives the tensors the backward needs.
    Returns (out [b*sq, h] fp32, am_out)."""
    (g1, b1, wqkv, bqkv, wd, bd, g3, b3, g2, b2, w1, bb1, w2, bb2, g4, b4) = P
    h = x.shape[1]
    training = save is not None
    scal = ops.new_scalars(4, x.device)
    ln1, mean1, rstd1 = ops.layernorm_absmax_fwd(x, am_x, g1, b1, eps, save_stats=training)
    qkv = ops.gemm(ln1, wqkv, bias=bqkv)
    qkv3 = qkv.view(b, sq, 3 * h)
    q, k, v = qkv3[..., :h], qkv3[..., h:2 * h], qkv3[..., 2 * h:]
    if kv is not None:
        k, v = kv(k, v)
    if attn is not None:            # sparse inference: attention over a gathered key set
        ctx, lse = attn(q), None
    elif isinstance(sep, SparseSpec):   # sparse training: causal band + gathered pivots, one softmax
        sp = (q, k, v, heads, sep.pivot_idx, sep.w, sep.times)
        if training and drops is not None and drops['attn'][0] > 0:
            ctx, lse, amask = ops.attn_sparse_fwd(*sp, want_lse=True, dropout=drops['attn'])
            drops['attn_mask'] = amask
        elif training:
            ctx, lse = ops.attn_sparse_fwd(*sp, want_lse=True)
        elif drops is not None and drops['attn'][0] > 0:   # forward only (checkpointed pass): same site, mask not kept
            ctx, _ = ops.attn_sparse_fwd(*sp, dropout=drops['attn'])
            lse = None
        else:
            ctx, lse = ops.attn_sparse_fwd(*sp), None
    elif training and drops is not None and drops['attn'][0] > 0:
        ctx, lse, amask = ops.attn_fwd(q, k, v, heads, sep=sep, want_lse=True, dropout=drops['attn'])
        drops['attn_mask'] = amask
    elif training:
        ctx, lse = ops.attn_fwd(q, k, v, heads, sep=sep, want_lse=True)
    elif drops is not None and drops['attn'][0] > 0:   # forward only (checkpointed pass): same sites, masks not kept
        ctx, _ = ops.attn_fwd(q, k, v, heads, sep=sep, dropout=drops['attn'])
        lse = None
    else:
        ctx, lse = ops.attn_fwd(q, k, v, heads, sep=sep), None
    ctx2 = ctx.view(b * sq, h)
    d_out_site = drops['out'] if drops is not None else None
    d_mlp_site = drops['mlp'] if drops is not None else None
    attn_out = ops.gemm(ctx2, wd, bias=bd, absmax=scal[0:1], dropout=d_out_site)
    y, mean3, rstd3 = ops.layernorm_absmax_fwd(attn_out, scal[0:1], g3, b3, eps, residual=x, out_dtype=torch.float32,
                                               absmax_out=scal[1:2], save_stats=training)
    ln2, mean2, rstd2 = ops.layernorm_absmax_fwd(y, scal[1:2], g2, b2, eps, save_stats=training)
    if training:
        h4, pre = ops.gemm(ln2, w1, bias=bb1, act=ops.ACT_GELU, want_preact=True)
    else:
        h4, pre = ops.gemm(ln2, w1, bias=bb1, act=ops.ACT_GELU), None
    mlp_out = ops.gemm(h4, w2, bias=bb2, absmax=scal[2:3], dropout=d_mlp_site)
    out, mean4, rstd4 = ops.layernorm_absmax_fwd(mlp_out, scal[2:3], g4, b4, eps, residual=y, out_dtype=torch.float32,
                                                 absmax_out=scal[3:4], save_stats=training)
    if training:
        save.extend([x, ln1, qkv, ctx, lse, attn_out, y, ln2, pre, h4, mlp_out,
                     mean1, rstd1, mean2, rstd2, mean3, rstd3, mean4, rstd4])
    return out, scal[3:4]


def layer_backward(d_out, saved, P, heads, b, sq, sep, drops=None):
    """Backward of layer_forward.  d_out: [b*sq, h] fp32.  Returns (d_x fp32, 16 parameter gradients bf16)."""
    (x, ln1, qkv, ctx, lse, attn_out, y, ln2, pre, h4, mlp_out,
     mean1, rstd1, mean2, rstd2, mean3, rstd3, mean4, rstd4) = saved
    (g1, b1, wqkv, bqkv, wd, bd, g3, b3, g2, b2, w1, bb1, w2, bb2, g4, b4) = P
    h = x.shape[1]
    M = b * sq
    # out = y + LN4(mlp_out)
    fuse_bias = h % 256 == 0          # the fused LN backward also returns the column sums of dx = the bias gradient
    r4 = ops.layernorm_absmax_bwd(mlp_out, d_out, mean4, rstd4, g4, dx_dtype=torch.bfloat16,
                                  dropout=drops['mlp'] if drops else None, want_dxsum=fuse_bias)
    d_mlp_out, dg4, db4 = r4[:3]
    d_pre = ops.gemm(d_mlp_out, w2, b_mn_major=True, act=ops.ACT_GELU_GRAD, aux=pre)   # (dY W2) * gelu'(pre)
    dw2 = ops.gemm(d_mlp_out, h4, a_mn_major=True, b_mn_major=True)
    dbb2 = r4[3] if fuse_bias else ops.colsum(d_mlp_out)
    d_ln2 = ops.gemm(d_pre, w1, b_mn_major=True)
    dw1 = ops.gemm(d_pre, ln2, a_mn_major=True, b_mn_major=True)
    dbb1 = ops.colsum(d_pre)
    d_y, dg2, db2 = ops.layernorm_absmax_bwd(y, d_ln2, mean2, rstd2, g2, dres=d_out, dx_dtype=torch.float32)
    # y = x + LN3(attn_out)
    r3 = ops.layernorm_absmax_bwd(attn_out, d_y, mean3, rstd3, g3, dx_dtype=torch.bfloat16,
                                  dropout=drops['out'] if drops else None, want_dxsum=fuse_bias)
    d_attn_out, dg3, db3 = r3[:3]
    ctx2 = ctx.view(M, h)
    d_ctx = ops.gemm(d_attn_out, wd, b_mn_major=True)
    dwd = ops.gemm(d_attn_out, ctx2, a_mn_major=True, b_mn_major=True)
    dbd = r3[3] if fuse_bias else ops.colsum(d_attn_out)
    qkv3 = qkv.view(b, sq, 3 * h)
    use_ad = bool(drops) and drops['attn'][0] > 0
    if isinstance(sep, SparseSpec):
        d_qkv = ops.attn_sparse_bwd(qkv3[..., :h], qkv3[..., h:2 * h], qkv3[..., 2 * h:], ctx, d_ctx.view(b, sq, h), lse,
                                    heads, sep.pivot_idx, sep.w, sep.times, dropout_p=drops['attn'][0] if use_ad else 0.0,
                                    drop_mask=drops['attn_mask'] if use_ad else None)
    else:
        d_qkv = ops.attn_bwd(qkv3[..., :h], qkv3[..., h:2 * h], qkv3[..., 2 * h:], ctx, d_ctx.view(b, sq, h), lse, heads,
                             sep=sep, dropout_p=drops['attn'][0] if use_ad else 0.0,
                             drop_mask=drops['attn_mask'] if use_ad else None)
    d_qkv2 = d_qkv.view(M, 3 * h)
    d_ln1 = ops.gemm(d_qkv2, wqkv, b_mn_major=True)
    dwqkv = ops.gemm(d_qkv2, ln1, a_mn_major=True, b_mn_major=True)
    dbqkv = ops.colsum(d_qkv2)
    d_x, dg1, db1 = ops.layernorm_absmax_bwd(x, d_ln1, mean1, rstd1, g1, dres=d_y, dx_dtype=torch.float32)
    return d_x, (dg1, db1, dwqkv, dbqkv, dwd, dbd, dg3, db3, dg2, db2, dw1, dbb1, dw2, dbb2, dg4, db4)


class _LayerFn(torch.autograd.Function):
    """autograd wrapper of layer_forward / layer_backward (training path, no memory)."""

    @staticmethod
    def forward(ctx, x, am_x, heads, eps, b, sq, sep, p_attn, p_out, *params):
        P = tuple(_as_bf16(p) for p in params)
        save = []
        drops = None
        if p_attn > 0 or p_out > 0:   # three dropout sites per layer: attention probs, attention output, MLP output
            sa, so, sm = next_dropout_site(), next_dropout_site(), next_dropout_site()
            drops = {'attn': (p_attn, sa[0], sa[1]), 'out': (p_out, so[0], so[1]), 'mlp': (p_out, sm[0], sm[1])}
        out, am_out = layer_forward(x, am_x, P, heads, eps, b, sq, sep, save=save, drops=drops)
        amask = drops.pop('attn_mask', None) if drops else None
        ctx.drops = drops
        ctx.has_amask = amask is not None
        if amask is not None:
            save.append(amask)
        ctx.save_for_backward(*save, *P)
        ctx.cfg = (heads, b, sq, sep, tuple(p.dtype for p in params))
        ctx.mark_non_differentiable(am_out)
        return out, am_out

    @staticmethod
    def backward(ctx, d_out, _d_am):
        heads, b, sq, sep, pdt = ctx.cfg
        saved = ctx.saved_tensors
        n = len(saved) - 16
        drops = ctx.drops
        acts = saved[:n]
        if ctx.has_amask:
            drops = dict(drops, attn_mask=saved[n - 1])
            acts = saved[:n - 1]
        d_x, grads = layer_backward(d_out.contiguous(), acts, saved[n:], heads, b, sq, sep, drops=drops)
        grads = tuple(g if g.dtype == dt else g.to(dt) for g, dt in zip(grads, pdt))
        return (d_x, None, None, None, None, None, None, None, None) + grads


# ----------------------------------------------------------------------------------------------------
# modules
# ----------------------------------------------------------------------------------------------------
class GPT2ParallelSelfAttention(torch.nn.Module):
    """mpu/sparse_transformer.py:46-169 (same constructor, parameters `query_key_value`, `dense`)."""

    def __init__(self, hidden_size, num_attention_heads, attention_dropout_prob, output_dropout_prob, init_method,
                 output_layer_init_method=None, query_window=128, key_window_times=6):
        super().__init__()
        if output_layer_init_method is None:
            output_layer_init_method = init_method
        self.hidden_size_per_partition = hidden_size
        self.hidden_size_per_attention_head = divide(hidden_size, num_attention_heads)
        self.num_attention_heads_per_partition = num_attention_heads
        self.query_window = query_window
        self.key_window_times = key_window_times
        self.query_key_value = ColumnParallelLinear(hidden_size, 3 * hidden_size, stride=3, gather_output=False,
                                                    init_method=init_method)
        self.attention_dropout = torch.nn.Dropout(attention_dropout_prob)
        self.dense = RowParallelLinear(hidden_size, hidden_size, input_is_parallel=True,
                                       init_method=output_layer_init_method)
        self.output_dropout = torch.nn.Dropout(output_dropout_prob)

    def forward(self, hidden_states, ltor_mask, pivot_idx=None, is_sparse=0, mem=None):
        """Standalone (unfused) use: hidden_states [b, s, h] already layer-normed; inference only for mem.
        is_sparse == 1 (mpu/sparse_transformer.py:150-151): `ltor_mask` is the reference's pivot_attention_mask
        (rmask gathered at pivot_idx, :569) — the kernel evaluates that mask in closed form from pivot_idx."""
        if is_sparse not in (0, 1):
            raise NotImplementedError('is_sparse=2 runs through GPT2ParallelTransformer (K|V cache + cv_attn_gather)')
        b, sq, h = hidden_states.shape
        heads = self.num_attention_heads_per_partition
        src = hidden_states if mem is None else torch.cat((mem, hidden_states), 1)
        mixed = self.query_key_value(src)
        sk = src.shape[1]
        if is_sparse == 1:
            if mem is not None or pivot_idx is None:
                raise ValueError('sparse training attention needs pivot_idx and no memory')
            sep = SparseSpec(pivot_idx, self.query_window, self.key_window_times)
        else:
            sep = mask_to_sep(ltor_mask, sq, sk)
        mixed = _as_bf16(mixed)
        q = mixed[:, sk - sq:, :h]
        ctx = _AttnFn.apply(q, mixed[..., h:2 * h], mixed[..., 2 * h:], heads, sep)
        out = self.dense(ctx.to(hidden_states.dtype))
        return self.output_dropout(out)


class _AttnFn(torch.autograd.Function):
    """dropout: None or (p, seed, site) of the attention-probability dropout (sparse mode only)."""

    @staticmethod
    def forward(ctx, q, k, v, heads, sep, dropout=None):
        mask = None
        if isinstance(sep, SparseSpec) and dropout is not None:
            out, lse, mask = ops.attn_sparse_fwd(q, k, v, heads, sep.pivot_idx, sep.w, sep.times, want_lse=True,
                                                 dropout=dropout)
        elif isinstance(sep, SparseSpec):
            out, lse = ops.attn_sparse_fwd(q, k, v, heads, sep.pivot_idx, sep.w, sep.times, want_lse=True)
        else:
            out, lse = ops.attn_fwd(q, k, v, heads, sep=sep, want_lse=True)
        if mask is not None:
            ctx.save_for_backward(q, k, v, out, lse, mask)
        else:
            ctx.save_for_backward(q, k, v, out, lse)
        ctx.cfg = (heads, sep, dropout[0] if mask is not None else 0.0)
        return out

    @staticmethod
    def backward(ctx, d_out):
        q, k, v, out, lse = ctx.saved_tensors[:5]
        heads, sep, p_drop = ctx.cfg
        if q.shape[1] != k.shape[1]:
            raise NotImplementedError('attention backward with memory (sq != sk) is not supported')
        if isinstance(sep, SparseSpec):
            d_qkv = ops.attn_sparse_bwd(q, k, v, out, _as_bf16(d_out).contiguous(), lse, heads, sep.pivot_idx, sep.w,
                                        sep.times, dropout_p=p_drop,
                                        drop_mask=ctx.saved_tensors[5] if p_drop > 0 else None)
        else:
            d_qkv = ops.attn_bwd(q, k, v, out, _as_bf16(d_out).contiguous(), lse, heads, sep=sep)
        h = q.shape[2]
        return d_qkv[..., :h], d_qkv[..., h:2 * h], d_qkv[..., 2 * h:], None, None, None


@torch.jit.ignore
def gelu(x):
    """mpu/sparse_transformer.py:172-179."""
    return 0.5 * x * (1.0 + torch.tanh(0.7978845608028654 * x * (1.0 + 0.044715 * x * x)))


class GPT2ParallelMLP(torch.nn.Module):
    """mpu/sparse_transformer.py:189-234."""

    def __init__(self, hidden_size, output_dropout_prob, init_method, output_layer_init_method=None):
        super().__init__()
        if output_layer_init_method is None:
            output_layer_init_method = init_method
        self.dense_h_to_4h = ColumnParallelLinear(hidden_size, 4 * hidden_size, gather_output=False,
                                                  init_method=init_method)
        self.dense_4h_to_h = RowParallelLinear(4 * hidden_size, hidden_size, input_is_parallel=True,
                                               init_method=output_layer_init_method)
        self.dropout = torch.nn.Dropout(output_dropout_prob)

    def forward(self, hidden_states):
        return self.dropout(self.dense_4h_to_h(gelu(self.dense_h_to_4h(hidden_states))))


class GPT2ParallelTransformerLayer(torch.nn.Module):
    """mpu/sparse_transformer.py:237-342.  `forward` keeps the reference signature; the stack driver calls
    `fused_forward` on the fp32 residual stream."""

    def __init__(self, hidden_size, num_attention_heads, attention_dropout_prob, output_dropout_prob,
                 layernorm_epsilon, init_method, output_layer_init_method=None, query_window=128, key_window_times=6,
                 scale_normalization=True):
        super().__init__()
        if output_layer_init_method is None:
            output_layer_init_method = init_method
        if not scale_normalization:
            raise NotImplementedError('CogView always uses Sandwich-LN (scale_normalization=True)')
        self.hidden_size = hidden_size
        self.num_attention_heads = num_attention_heads
        self.layernorm_epsilon = layernorm_epsilon
        self.attention_dropout_prob = attention_dropout_prob
        self.output_dropout_prob = output_dropout_prob
        self.input_layernorm = LayerNorm(hidden_size, eps=layernorm_epsilon)
        self.attention = GPT2ParallelSelfAttention(hidden_size, num_attention_heads, attention_dropout_prob,
                                                   output_dropout_prob, init_method,
                                                   output_layer_init_method=output_layer_init_method,
                                                   query_window=query_window, key_window_times=key_window_times)
        self.post_attention_layernorm = LayerNorm(hidden_size, eps=layernorm_epsilon)
        self.scale_normalization = scale_normalization
        self.third_layernorm = LayerNorm(hidden_size, eps=layernorm_epsilon)
        self.fourth_layernorm = LayerNorm(hidden_size, eps=layernorm_epsilon)
        self.mlp = GPT2ParallelMLP(hidden_size, output_dropout_prob, init_method,
                                   output_layer_init_method=output_layer_init_method)

    def param_list(self):
        sd = dict(self.named_parameters())
        return [sd[n] for n in _PARAM_ORDER]

    def fused_forward(self, x, am_x, b, sq, sep, kv=None, attn=None):
        """x: fp32 [b*sq, h] residual stream, am_x: max|x| scalar tensor -> (out, am_out)."""
        params = self.param_list()
        if torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in params)):
            if kv is not None:
                raise NotImplementedError('training with memory is not supported')
            p_attn = self.attention_dropout_prob if self.training else 0.0
            p_out = self.output_dropout_prob if self.training else 0.0
            return _LayerFn.apply(x, am_x, self.num_attention_heads, self.layernorm_epsilon, b, sq, sep, p_attn, p_out,
                                  *params)
        drops = None
        if self.training and (self.attention_dropout_prob > 0 or self.output_dropout_prob > 0):
            # training-mode forward without autograd (the first pass of mpu.checkpoint): draw the same three sites
            sa, so, sm = next_dropout_site(), next_dropout_site(), next_dropout_site()
            drops = {'attn': (self.attention_dropout_prob, sa[0], sa[1]), 'out': (self.output_dropout_prob, so[0], so[1]),
                     'mlp': (self.output_dropout_prob, sm[0], sm[1])}
        P = tuple(_as_bf16(p.detach()) for p in params)
        return layer_forward(x, am_x, P, self.num_attention_heads, self.layernorm_epsilon, b, sq, sep, kv=kv, attn=attn,
                             drops=drops)

    def forward(self, hidden_states, ltor_mask, pivot_idx=None, is_sparse=0, mem=None):
        """Reference signature: hidden_states [b, s, h], mask [1,1,s,s] or int sep; `mem` = hidden-state memory
        [b, t, h] (re-normalised and re-projected exactly like mpu/sparse_transformer.py:320, :136-141).
        is_sparse == 1: `ltor_mask` is the pivot_attention_mask of :569 (evaluated in closed form from pivot_idx)."""
        if is_sparse not in (0, 1):
            raise NotImplementedError('is_sparse=2 runs through GPT2ParallelTransformer (K|V cache + cv_attn_gather)')
        b, sq, h = hidden_states.shape
        x = hidden_states.reshape(b * sq, h).float().contiguous()
        am_x = ops.absmax(x)
        if is_sparse == 1:
            if mem is not None or pivot_idx is None:
                raise ValueError('sparse training attention needs pivot_idx and no memory')
            att = self.attention
            out, _ = self.fused_forward(x, am_x, b, sq, SparseSpec(pivot_idx, att.query_window, att.key_window_times))
        elif mem is None:
            sep = mask_to_sep(ltor_mask, sq, sq)
            out, _ = self.fused_forward(x, am_x, b, sq, sep)
        else:
            t = mem.shape[1]
            sep = mask_to_sep(ltor_mask, sq, sq + t)
            P = tuple(_as_bf16(p.detach()) for p in self.param_list())
            memf = mem.reshape(b * t, h).float().contiguous()
            ln_mem, _, _ = ops.layernorm_absmax_fwd(memf, ops.absmax(memf), P[0], P[1], self.layernorm_epsilon)
            kv_mem = ops.gemm(ln_mem, P[2][h:], bias=P[3][h:]).view(b, t, 2 * h)   # K,V of the memory

            def kv(k_new, v_new):
                kvc = torch.cat((kv_mem, torch.cat((k_new, v_new), dim=-1)), dim=1)
                return kvc[..., :h], kvc[..., h:]
            out, _ = self.fused_forward(x, am_x, b, sq, sep, kv=kv)
        return out.view(b, sq, h).to(hidden_states.dtype)


def unscaled_init_method(sigma):
    """N(0, sigma) — mpu/sparse_transformer.py:344-349."""
    def init_(tensor):
        return torch.nn.init.normal_(tensor, mean=0.0, std=sigma)
    return init_


def scaled_init_method(sigma, num_layers):
    """N(0, sigma / sqrt(2 * num_layers)) — mpu/sparse_transformer.py:352-358."""
    std = sigma / math.sqrt(2.0 * num_layers)

    def init_(tensor):
        return torch.nn.init.normal_(tensor, mean=0.0, std=std)
    return init_


class _EmbedFn(torch.autograd.Function):
    """hidden = wte[ids] + wpe[pos] as one gather kernel (fp32 out + its abs-max); scatter-add backward."""

    @staticmethod
    def forward(ctx, ids, pos, wte, wpe, p_drop=0.0):
        am = ops.new_scalars(1, wte.device)
        wb, pb = _as_bf16(wte), _as_bf16(wpe)
        ctx.drop = None
        if p_drop > 0:
            seed, site = next_dropout_site()
            ctx.drop = (p_drop, seed, site)
        out = ops.embed_fwd(ids, pos, wb.contiguous(), pb.contiguous(), am, dropout=ctx.drop)
        ctx.save_for_backward(ids, pos)
        ctx.meta = (wte.shape, wpe.shape, wte.dtype, wpe.dtype, wte.device)
        ctx.mark_non_differentiable(am)
        return out, am

    @staticmethod
    def backward(ctx, d_out, _d_am):
        ids, pos = ctx.saved_tensors
        ws, ps, wdt, pdt, dev = ctx.meta
        dwte = torch.zeros(ws, dtype=torch.bfloat16, device=dev)
        dwpe = torch.zeros(ps, dtype=torch.bfloat16, device=dev)
        ops.embed_bwd(ids, pos, d_out.contiguous(), dwte, dwpe, dropout=ctx.drop)
        return None, None, dwte.to(wdt), dwpe.to(pdt), None


class GPT2ParallelTransformer(torch.nn.Module):
    """mpu/sparse_transformer.py:361-626 (same constructor; parameters `position_embeddings`, `layers.N.*`,
    `final_layernorm`)."""

    def __init__(self, num_layers, hidden_size, num_attention_heads, max_sequence_length, max_memory_length,
                 embedding_dropout_prob, attention_dropout_prob, output_dropout_prob, checkpoint_activations,
                 checkpoint_num_layers=1, layernorm_epsilon=1.0e-5, init_method_std=0.02,
                 use_scaled_init_for_output_weights=True, query_window=128, key_window_times=6, num_pivot=768):
        super().__init__()
        self.checkpoint_activations = checkpoint_activations
        self.checkpoint_num_layers = checkpoint_num_layers
        self.max_memory_length = max_memory_length
        self.max_sequence_length = max_sequence_length
        self.hidden_size = hidden_size
        self.num_attention_heads = num_attention_heads
        self.embedding_dropout_prob = embedding_dropout_prob
        output_layer_init_method = None
        if use_scaled_init_for_output_weights:
            output_layer_init_method = scaled_init_method(init_method_std, num_layers)
        self.embedding_dropout = torch.nn.Dropout(embedding_dropout_prob)
        self.position_embeddings = torch.nn.Embedding(max_sequence_length, hidden_size)
        torch.nn.init.normal_(self.position_embeddings.weight, mean=0.0, std=init_method_std)
        self.query_window = query_window
        self.key_window_times = key_window_times
        self.num_pivot = num_pivot
        self.layers = torch.nn.ModuleList([
            GPT2ParallelTransformerLayer(hidden_size, num_attention_heads, attention_dropout_prob,
                                         output_dropout_prob, layernorm_epsilon, unscaled_init_method(init_method_std),
                                         output_layer_init_method=output_layer_init_method, query_window=query_window,
                                         key_window_times=key_window_times, scale_normalization=True)
            for _ in range(num_layers)])
        self.final_layernorm = LayerNorm(hidden_size, eps=layernorm_epsilon)
        self.rmask = None
        # 'hidden': mems are the reference's per-layer hidden states (exact semantics, O(t h^2) per step);
        # 'kv'    : mems are per-layer K|V caches [b, t, 2h] (same list length and batch/time axes)
        self.mems_mode = os.environ.get('COGVIEW_B200_MEMS', 'kv')
        self._kv = None

    # -- the stack on the fp32 residual stream ---------------------------------------------------------
    def sparse_index_plan(self, key_length, txt_indices_bool, img_indices_bool, b, device):
        """Index bookkeeping of is_sparse == 2 (mpu/sparse_transformer.py:498-520): trailing window, text / image
        positions before it, and the pivot count."""
        w, times = self.query_window, self.key_window_times
        left_boundary = max(0, key_length - times * w)
        window_idx = torch.arange(left_boundary, key_length, device=device, dtype=torch.long).expand(b, -1)
        img_indices = [img_indices_bool[i][:left_boundary].nonzero(as_tuple=False).view(-1) for i in range(b)]
        txt_indices = [txt_indices_bool[i][:left_boundary].nonzero(as_tuple=False).view(-1) for i in range(b)]
        ratio = self.num_pivot / self.max_sequence_length
        max_text_num = max(len(t) for t in txt_indices)
        num_pivot = max_text_num + int((left_boundary - max_text_num) * ratio)
        return window_idx, img_indices, txt_indices, num_pivot

    @staticmethod
    def sample_pivot_idx(img_indices, txt_indices, num_pivot):
        """:557-565 / :591-599 — all text positions + a Python random.sample of image positions, per sequence."""
        return torch.stack([
            torch.cat((text_idx,
                       img_indices[i][torch.tensor(random.sample(range(len(img_indices[i])), k=num_pivot - len(text_idx)),
                                                   dtype=torch.long, device=text_idx.device)]), dim=0)
            for i, text_idx in enumerate(txt_indices)])

    def sample_pivots(self, window_idx, img_indices, txt_indices, num_pivot):
        """Fresh pivots for one layer of sparse inference (:591-600) followed by the trailing window."""
        return torch.cat((GPT2ParallelTransformer.sample_pivot_idx(img_indices, txt_indices, num_pivot), window_idx),
                         dim=-1)

    def run_layers(self, x, am_x, b, sq, sep, mems, word_embedding_weight=None, is_sparse=0, txt_indices_bool=None,
                   img_indices_bool=None):
        """x fp32 [b*sq, h].  Returns (final-LN output bf16 [b*sq, h], mem_layers list)."""
        from . import kv_cache
        h = self.hidden_size
        keep_mems = self.max_memory_length > 0
        mode = self.mems_mode if keep_mems else None
        if mems and torch.is_grad_enabled() and x.requires_grad:
            raise NotImplementedError('training with memory is not supported')
        if mode == 'kv' and torch.is_grad_enabled() and x.requires_grad:
            mode = 'hidden'   # training forward: return the reference's detached hidden-state mems
        hidden_mems = [x.detach().view(b, sq, h)] if mode == 'hidden' else []
        caches = kv_cache.prepare(self, mems, b, sq) if mode == 'kv' else None
        plan = None
        if is_sparse == 2:
            if mode != 'kv' or torch.is_grad_enabled():
                raise NotImplementedError("is_sparse=2 (sparse inference) needs max_memory_length > 0, mems_mode 'kv' "
                                          "and torch.no_grad()")
            if sq > self.query_window * self.key_window_times:
                raise ValueError('the fed tokens must fit in the attention window (query_window * key_window_times)')
            plan = self.sparse_index_plan(caches.t + sq, txt_indices_bool, img_indices_bool, b, x.device)
        elif is_sparse == 1:
            # sparse training (mpu/sparse_transformer.py:491-496, :556-589): fresh pivots for every checkpointed chunk
            if mems:
                raise NotImplementedError('sparse training attention takes no memory (:567 asserts the same)')
            if not self.checkpoint_activations:
                raise AssertionError('Please use checkpoint_activations for sparse attention training.')   # :586
            if sq % self.query_window != 0:
                raise ValueError('The seq_len must be exactly divided by window_size.')                       # :713
            img_all = [img_indices_bool[i][:sq].nonzero(as_tuple=False).view(-1) for i in range(b)]
            txt_all = [txt_indices_bool[i][:sq].nonzero(as_tuple=False).view(-1) for i in range(b)]
        elif is_sparse != 0:
            raise ValueError('is_sparse must be 0, 1 or 2')
        spec = None
        for i, layer in enumerate(self.layers):
            if is_sparse == 1 and i % max(1, self.checkpoint_num_layers) == 0:
                spec = SparseSpec(self.sample_pivot_idx(img_all, txt_all, self.num_pivot), self.query_window,
                                  self.key_window_times)
            if spec is not None:
                sep = spec
            if mode == 'kv' and plan is not None:
                pw_idx = self.sample_pivots(*plan)
                cache_i, t_all, heads = caches.buf[i], caches.t + sq, self.num_attention_heads

                def gather_attn(q, cache_i=cache_i, pw_idx=pw_idx):
                    return ops.attn_gather(q, cache_i[:, :t_all], pw_idx, heads)
                out, am_x = layer.fused_forward(x, am_x, b, sq, sep, kv=caches.appender(i), attn=gather_attn)
            elif mode == 'kv':
                out, am_x = layer.fused_forward(x, am_x, b, sq, sep, kv=caches.appender(i))
            elif mems:   # hidden-state memory: exact reference semantics
                out = layer(x.view(b, sq, h), sep, mem=mems[i]).view(b * sq, h)
                am_x = ops.absmax(out)
            elif self.checkpoint_activations and torch.is_grad_enabled() and x.requires_grad:
                def run(x_, am_, layer=layer, sep=sep):      # `sep` bound now: the recomputation runs in the backward
                    return layer.fused_forward(x_, am_, b, sq, sep)
                out, am_x = checkpoint(run, x, am_x)
            else:
                out, am_x = layer.fused_forward(x, am_x, b, sq, sep)
            x = out
            if mode == 'hidden':
                hidden_mems.append(x.detach().view(b, sq, h))
        fl = self.final_layernorm
        if torch.is_grad_enabled() and (x.requires_grad or fl.weight.requires_grad):
            y = _FinalLNFn.apply(x, am_x, fl.weight, fl.bias, fl.eps)
        else:
            y, _, _ = ops.layernorm_absmax_fwd(x, am_x, _as_bf16(fl.weight.detach()), _as_bf16(fl.bias.detach()),
                                               fl.eps)
        if mode == 'hidden':
            mem_layers = self.update_mems(hidden_mems, mems)
        elif mode == 'kv':
            mem_layers = caches.views()
        else:
            mem_layers = []
        return y, mem_layers

    def forward(self, hidden_states, position_ids, attention_mask, txt_indices_bool, img_indices_bool, is_sparse=0,
                *mems):
        """Reference signature (mpu/sparse_transformer.py:471): hidden_states = word embeddings [b, s, h].
        Returns (final-LN output [b, s, h], *mems)."""
        b, sq, h = hidden_states.shape
        mem_len = mems[0].size(1) if mems else 0
        sep = 0 if is_sparse != 0 else mask_to_sep(attention_mask, sq, sq + mem_len)
        pe = torch.nn.functional.embedding(position_ids, self.position_embeddings.weight)
        x = (hidden_states.float() + pe.float()).reshape(b * sq, h).contiguous()
        if self.training and self.embedding_dropout_prob > 0:
            x = torch.nn.functional.dropout(x, self.embedding_dropout_prob)   # standalone entry (GPT2Model fuses it)
        am_x = ops.absmax(x.detach())
        y, mem_layers = self.run_layers(x, am_x, b, sq, sep, mems, is_sparse=is_sparse,
                                        txt_indices_bool=txt_indices_bool, img_indices_bool=img_indices_bool)
        return (y.view(b, sq, h).to(hidden_states.dtype), *mem_layers)

    def update_mems(self, hiddens, mems):
        """mpu/sparse_transformer.py:615-626."""
        memory_length = mems[0].size(1) if mems else 0
        query_length = hiddens[0].size(1)
        new_memory_length = min(self.max_memory_length, memory_length + query_length)
        new_mems = []
        with torch.no_grad():
            for i in range(len(hiddens)):
                if new_memory_length <= query_length:
                    new_mems.append(hiddens[i][:, -new_memory_length:])
                else:
                    new_mems.append(torch.cat((mems[i][:, -new_memory_length + query_length:].to(hiddens[i].dtype),
                                               hiddens[i]), dim=1))
        return new_mems


class _FinalLNFn(torch.autograd.Function):
    """Final LayerNorm on the fp32 stream -> bf16 (feeds the logits GEMM)."""

    @staticmethod
    def forward(ctx, x, am_x, weight, bias, eps):
        w = _as_bf16(weight)
        y, mean, rstd = ops.layernorm_absmax_fwd(x, am_x, w, _as_bf16(bias), eps, save_stats=True)
        ctx.save_for_backward(x, mean, rstd, w)
        ctx.meta = (weight.dtype, bias.dtype)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, mean, rstd, w = ctx.saved_tensors
        dx, dg, db = ops.layernorm_absmax_bwd(x, _as_bf16(dy).contiguous(), mean, rstd, w, dx_dtype=torch.float32)
        return dx, None, dg.to(ctx.meta[0]), db.to(ctx.meta[1]), None


def sparse_attention(q, k, v, pivot_idx, pivot_attention_mask=None, query_window=128, key_window_times=6,
                     attention_dropout=None):
    """mpu/sparse_transformer.py:675-725 on [b, np, s, hn] tensors (API parity; the model path reads the packed QKV
    GEMM output in place).  `pivot_attention_mask` is accepted for signature parity: the kernel evaluates the mask the
    reference builds (rmask of :491-496 gathered at pivot_idx, :569) in closed form — pivot p is visible to query i
    iff pivot_idx[p] < band_start(i).  An `attention_dropout` module in training mode applies its p to the joint
    softmax inside the kernel (counter-based keep bits, seed drawn from torch's generator as in standard_attention;
    the reference draws from the model-parallel RNG tracker, :719-721).  Differentiable."""
    b, nh, s, hn = q.shape

    def tok_major(t):
        return _as_bf16(t).permute(0, 2, 1, 3).reshape(b, t.shape[2], nh * hn).contiguous()

    drop = None
    if attention_dropout is not None and attention_dropout.training and attention_dropout.p > 0:
        drop = (float(attention_dropout.p), int(torch.randint(0, 2 ** 62, (1,)).item()), 0)
    ctx = _AttnFn.apply(tok_major(q), tok_major(k), tok_major(v), nh, SparseSpec(pivot_idx, query_window, key_window_times),
                        drop)
    return ctx.view(b, s, nh, hn).permute(0, 2, 1, 3).to(q.dtype)


def sparse_attention_inference(q, k, v, pivot_and_window_idx, **kwargs):
    """mpu/sparse_transformer.py:727-750 on [b, np, s, hn] tensors (API parity; the model path reads the K|V cache in
    place): dense softmax over K[idx], V[idx] with the causal fix for the trailing queries."""
    b, nh, sq, hn = q.shape
    sk = k.shape[2]
    kv = torch.cat((_as_bf16(k).permute(0, 2, 1, 3).reshape(b, sk, nh * hn),
                    _as_bf16(v).permute(0, 2, 1, 3).reshape(b, sk, nh * hn)), dim=-1).contiguous()
    qt = _as_bf16(q).permute(0, 2, 1, 3).reshape(b, sq, nh * hn).contiguous()
    ctx = ops.attn_gather(qt, kv, pivot_and_window_idx, nh)
    return ctx.view(b, sq, nh, hn).permute(0, 2, 1, 3).to(q.dtype)
