"""CPU fp32 restatement of sparse TRAINING attention WITH attention-probability dropout (mpu/sparse_transformer.py:675-725,
the dropout of :719-721), for parity runs under a given keep tensor.

oracle/cogview_oracle.py restates the reference with dropout off.  The functions here follow its sparse_attention and
transformer_layer operation for operation and add one step: the joint softmax probabilities are multiplied by
keep / (1 - p) before the two products.  With an all-ones keep tensor and p = 0 they reproduce cogview_oracle bit for
bit (tests/test_sparse_dropout_cpu.py checks that).  They are pinned to the unmodified reference through
tests/golden/sparse_dropout.npz (oracle/make_sparse_dropout_golden.py).

keep: 0/1 tensor in the reference's own joint layout [b, np, s, n_piv + w*times]: pivots in pivot_idx order, then the
window slots of _chunk (:629-650); slot t of query i is key (i // w - times + 1) * w + t."""
import math

import torch
import torch.nn.functional as F

from oracle import cogview_oracle as O


def sparse_attention(q, k, v, pivot_idx, pivot_attention_mask, query_window, key_window_times, keep, p):
    """O.sparse_attention with the joint probabilities multiplied by keep / (1 - p)."""
    b, n_head, s, hn = q.shape
    n_piv = pivot_idx.shape[1]
    w, times = query_window, key_window_times
    gidx = pivot_idx.view(b, 1, n_piv, 1).expand(b, n_head, n_piv, hn)
    pk, pv = torch.gather(k, 2, gidx), torch.gather(v, 2, gidx)
    pm = pivot_attention_mask.unsqueeze(1)
    sp = torch.matmul(q, pk.transpose(-1, -2)) * (pm / math.sqrt(hn)) - 10000.0 * (1.0 - pm)
    sp = sp + math.log(s // n_piv)
    if s % w != 0:
        raise ValueError('The seq_len must be exactly divided by window_size.')
    wk, wv = O._overlapping_windows(k, w, times), O._overlapping_windows(v, w, times)
    wq = q.view(b, n_head, s // w, w, hn)
    sw = torch.matmul(wq, wk.transpose(-1, -2))
    wm = torch.ones((w, w * times), dtype=sw.dtype).tril_(diagonal=w * (times - 1))
    sw = sw * (wm / math.sqrt(hn)) - 10000.0 * (1.0 - wm)
    sw = sw.clone()
    for t in range(1, times):  # left padding of the first windows
        sw[:, :, t - 1, :, :w * times - w * t] -= 10000.0
    sw = sw.view(b, n_head, s, w * times)
    probs = torch.softmax(torch.cat((sp, sw), dim=-1), dim=-1)
    probs = probs * (keep / (1.0 - p))           # attention dropout on the joint probabilities (:719-721)
    ctx_p = torch.matmul(probs[..., :n_piv], pv)
    ctx_w = torch.einsum('bcgwk,bcgkh->bcgwh', probs[..., n_piv:].view(b, n_head, s // w, w, w * times), wv)
    return ctx_p + ctx_w.reshape(b, n_head, s, hn)


def transformer_layer(sd, i, x, pivot_attention_mask, n_heads, pivot_idx, query_window, key_window_times, keep, p):
    """O.transformer_layer(..., is_sparse=1) with the attention dropout above (output dropouts off)."""
    pre = 'transformer.layers.%d.' % i

    def ln(name, t):
        return O.layernorm_absmax(t, sd[pre + name + '.weight'], sd[pre + name + '.bias'])

    ln1 = ln('input_layernorm', x)
    ap = pre + 'attention.'
    mixed = F.linear(ln1, sd[ap + 'query_key_value.weight'], sd[ap + 'query_key_value.bias'])
    qm, km, vm = mixed.chunk(3, dim=-1)
    q, k, v = O._heads(qm, n_heads), O._heads(km, n_heads), O._heads(vm, n_heads)
    ctx = sparse_attention(q, k, v, pivot_idx, pivot_attention_mask, query_window, key_window_times, keep, p)
    bsz, _, sq, hn = ctx.shape
    ctx = ctx.permute(0, 2, 1, 3).reshape(bsz, sq, n_heads * hn)
    att = F.linear(ctx, sd[ap + 'dense.weight']) + sd[ap + 'dense.bias']
    y = x + ln('third_layernorm', att)
    m = O.mlp(sd, pre + 'mlp.', ln('post_attention_layernorm', y))
    return y + ln('fourth_layernorm', m)
