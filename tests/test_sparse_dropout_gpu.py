"""GPU: attention-probability dropout in sparse TRAINING attention (is_sparse = 1, mpu/sparse_transformer.py:675-725,
dropout on the joint softmax :719-721) — cv_attn_sparse_dropout_fwd / cv_attn_sparse_dropout_bwd and the layers above.

Bitwise parity with torch's generator is not defined; these tests pin the SEMANTICS: the keep bits the forward returns
(three regions, include/cogview_b200.h) agree between layouts on every visible entry, behave like independent
Bernoulli(1 - p) draws, and the outputs and gradients equal the oracle's autograd under exactly those keep bits mapped to
the reference's joint layout [b, nh, s, n_piv + w*times].  p = 0 through the new entry points is bitwise the existing
path.  Tolerances (bf16 tensor-core math vs the fp32 oracle): 2e-2 of the output scale, 4e-2 of each gradient's scale;
layer parity uses those of test_model_sparse_training_step_matches_oracle."""
import os
import random

import pytest
import torch

from oracle import recipes
from oracle import sparse_dropout_oracle as SD

pytestmark = pytest.mark.gpu
P = 0.1
SHAPES = [(2, 3, 512, 64, 3, 96, (48, 20)), (1, 2, 1024, 128, 6, 200, (64,)), (1, 2, 4096, 128, 6, 768, (100,)),
          (2, 1, 256, 128, 2, 40, (0, 7)), (1, 1, 768, 128, 6, 64, (30,))]


def _rmask(s, w, times):
    g = s // w
    tmp = torch.tril(1 - torch.block_diag(*torch.ones((g - times + 1, w, w))))
    return torch.nn.functional.pad(tmp, (0, (times - 1) * w, (times - 1) * w, 0))


def _pivots(b, s, n_piv, txt_n, seed):
    random.seed(seed)
    return torch.stack([
        torch.cat((torch.arange(0, txt_n[i]),
                   torch.tensor(random.sample(range(txt_n[i], s), n_piv - txt_n[i]), dtype=torch.long)))
        for i in range(b)])


def _band_start(i, w, times):
    return max(0, i // w - times + 1) * w


def _tile_lists(s, w, times, n_piv):
    """(jb0, nband, npt) per 128-query block and the longest list — the schedule of csrc/attention_fwd.cu."""
    npt = (n_piv + 127) // 128
    lists = []
    for qb in range((s + 127) // 128):
        q0, q_last = qb * 128, min(qb * 128 + 128, s) - 1
        jb0 = _band_start(q0, w, times) // 128
        lists.append((jb0, q_last // 128 - jb0 + 1, npt if _band_start(q_last, w, times) > 0 else 0))
    return lists, max(nb + npn for _, nb, npn in lists)


def _bits(words):
    sh = torch.arange(32, device=words.device, dtype=torch.int32)
    return ((words.unsqueeze(-1) >> sh) & 1).bool().flatten(-2)


def _decode(mask, b, nh, s, n_piv, w, times):
    """Keep bits from the three regions.  Returns (band_k, piv_k, band_q, piv_q, written_band, written_piv):
    band [b, nh, query, key], pivot [b, nh, query, pivot slot] from the key-major ([0], [1]) and the query-major ([2])
    regions; written_* [query, key / slot]: the tiles the query's block visits (the rest is never written)."""
    nqb, npt = (s + 127) // 128, (n_piv + 127) // 128
    S = nqb * 128
    lists, T = _tile_lists(s, w, times, n_piv)
    n0, n1 = b * nh * S * nqb * 4, b * nh * npt * 128 * nqb * 4
    m = mask.view(-1)
    assert m.numel() == n0 + n1 + b * nh * S * T * 4
    band_k = _bits(m[:n0].view(b, nh, S, nqb, 4)).view(b, nh, S, S).transpose(2, 3)
    piv_k = _bits(m[n0:n0 + n1].view(b, nh, npt * 128, nqb, 4)).view(b, nh, npt * 128, S).transpose(2, 3)
    qm = _bits(m[n0 + n1:].view(b, nh, S, T, 4))                     # [b, nh, query, T, 128]
    band_q = torch.zeros((b, nh, S, S), dtype=torch.bool, device=mask.device)
    piv_q = torch.zeros((b, nh, S, npt * 128), dtype=torch.bool, device=mask.device)
    wb = torch.zeros((S, S), dtype=torch.bool, device=mask.device)
    wp = torch.zeros((S, npt * 128), dtype=torch.bool, device=mask.device)
    for qb, (jb0, nb, npn) in enumerate(lists):
        r = slice(qb * 128, qb * 128 + 128)
        for j in range(nb):
            kt = jb0 + j
            band_q[:, :, r, kt * 128:kt * 128 + 128] = qm[:, :, r, j]
            wb[r, kt * 128:kt * 128 + 128] = True
        for t in range(npn):
            piv_q[:, :, r, t * 128:t * 128 + 128] = qm[:, :, r, nb + t]
            wp[r, t * 128:t * 128 + 128] = True
    return (band_k[..., :s, :s], piv_k[..., :s, :n_piv], band_q[..., :s, :s], piv_q[..., :s, :n_piv], wb[:s, :s],
            wp[:s, :n_piv])


def _visible(pivot_idx, s, w, times, device):
    """band [query, key] and pivot [b, query, slot] visibility of the sparse mask (closed form)."""
    i = torch.arange(s, device=device)
    bs = (torch.clamp(i // w - times + 1, min=0) * w)
    band = (i.view(1, -1) >= bs.view(-1, 1)) & (i.view(1, -1) <= i.view(-1, 1))
    piv = pivot_idx.to(device).unsqueeze(1) < bs.view(1, -1, 1)
    return band, piv


def _to_reference_layout(band_k, piv_k, s, w, times):
    """[b, nh, s, n_piv + w*times]: pivots in pivot_idx order, then the _chunk window slots (slot t of query i is key
    (i // w - times + 1) * w + t; left-padding slots get 1, their probability is 0 anyway)."""
    i = torch.arange(s, device=band_k.device).view(-1, 1)
    key = (i // w - times + 1) * w + torch.arange(w * times, device=band_k.device).view(1, -1)
    win = band_k.gather(-1, key.clamp(min=0).expand(band_k.shape[0], band_k.shape[1], -1, -1))
    win = win | (key < 0)
    return torch.cat((piv_k, win), dim=-1).float()


def _run(b, nh, s, w, times, n_piv, txt, dropout):
    from cogview_b200 import ops
    gen = torch.Generator().manual_seed(s + n_piv)
    h = nh * 64
    qkv = torch.randn((b, s, 3 * h), generator=gen).bfloat16()
    d_out = (torch.randn((b, s, h), generator=gen) * 0.5).bfloat16()
    pivot_idx = _pivots(b, s, n_piv, txt, seed=99)
    qc, pc = qkv.cuda(), pivot_idx.cuda()
    r = ops.attn_sparse_fwd(qc[..., :h], qc[..., h:2 * h], qc[..., 2 * h:], nh, pc, w, times, want_lse=True,
                            dropout=dropout)
    ctx, lse, mask = r if dropout is not None else (r[0], r[1], None)
    dqkv = ops.attn_sparse_bwd(qc[..., :h], qc[..., h:2 * h], qc[..., 2 * h:], ctx, d_out.cuda(), lse, nh, pc, w, times,
                               dropout_p=dropout[0] if dropout else 0.0, drop_mask=mask)
    torch.cuda.synchronize()
    return qkv, d_out, pivot_idx, ctx, lse, dqkv, mask


def test_p0_through_new_entry_points_is_bitwise_unchanged():
    from cogview_b200 import ops
    b, nh, s, w, times, n_piv, txt = SHAPES[1]
    qkv, d_out, pivot_idx, ctx, lse, dqkv, _ = _run(b, nh, s, w, times, n_piv, txt, None)
    h = nh * 64
    qc, pc, dc = qkv.cuda(), pivot_idx.cuda(), d_out.cuda()
    q, k, v = qc[..., :h], qc[..., h:2 * h], qc[..., 2 * h:]
    out = torch.empty_like(ctx)
    lse2 = torch.empty_like(lse)
    ws = torch.empty(ops.lib().cv_attn_sparse_workspace_bytes(b, nh, 64, n_piv), dtype=torch.uint8, device="cuda")
    ops.check(ops.lib().cv_attn_sparse_dropout_fwd(
        ops.ptr(q), q.stride(1), q.stride(0), ops.ptr(k), k.stride(1), k.stride(0), ops.ptr(v), v.stride(1), v.stride(0),
        ops.ptr(pc), ops.ptr(out), out.stride(1), out.stride(0), ops.ptr(lse2), ops.ptr(ws), b, nh, 64, s, n_piv, w, times,
        0.0, 0, 0, None, ops.stream_ptr()), "cv_attn_sparse_dropout_fwd")
    dqkv2 = torch.empty_like(dqkv)
    wsb = torch.empty(ops.lib().cv_attn_sparse_bwd_workspace_bytes(b, nh, 64, s, n_piv), dtype=torch.uint8,
                      device="cuda")
    ops.check(ops.lib().cv_attn_sparse_dropout_bwd(
        ops.ptr(q), q.stride(1), q.stride(0), ops.ptr(k), k.stride(1), k.stride(0), ops.ptr(v), v.stride(1), v.stride(0),
        ops.ptr(pc), ops.ptr(ctx), ops.ptr(dc), ops.ptr(lse), ops.ptr(dqkv2), ops.ptr(wsb), b, nh, 64, s, n_piv, w, times,
        0.0, None, ops.stream_ptr()), "cv_attn_sparse_dropout_bwd")
    torch.cuda.synchronize()
    assert torch.equal(out, ctx) and torch.equal(lse2, lse) and torch.equal(dqkv2, dqkv)
    # p > 0 without a keep-bit buffer is refused
    rc = ops.lib().cv_attn_sparse_dropout_fwd(
        ops.ptr(q), q.stride(1), q.stride(0), ops.ptr(k), k.stride(1), k.stride(0), ops.ptr(v), v.stride(1), v.stride(0),
        ops.ptr(pc), ops.ptr(out), out.stride(1), out.stride(0), ops.ptr(lse2), ops.ptr(ws), b, nh, 64, s, n_piv, w, times,
        0.1, 0, 0, None, ops.stream_ptr())
    assert rc != 0


@pytest.mark.parametrize("b,nh,s,w,times,n_piv,txt", SHAPES)
def test_sparse_dropout_forward_backward_match_oracle(b, nh, s, w, times, n_piv, txt):
    qkv, d_out, pivot_idx, ctx, lse, dqkv, mask = _run(b, nh, s, w, times, n_piv, txt, (P, 1234, 17))
    band_k, piv_k, band_q, piv_q, _, _ = _decode(mask, b, nh, s, n_piv, w, times)
    band_vis, piv_vis = _visible(pivot_idx, s, w, times, "cuda")
    assert torch.equal(band_k & band_vis, band_q & band_vis)                  # both layouts hold the same decisions
    pv = piv_vis.unsqueeze(1).expand(-1, nh, -1, -1)
    assert torch.equal(piv_k & pv, piv_q & pv)
    rate = band_k[:, :, band_vis].float().mean().item()
    assert abs(rate - (1 - P)) < 0.02
    keep = _to_reference_layout(band_k, piv_k, s, w, times).cpu()
    h = nh * 64

    def heads_first(t):
        return t.float().view(b, s, nh, 64).permute(0, 2, 1, 3).contiguous()
    q, k, v = (heads_first(qkv[..., i * h:(i + 1) * h]).requires_grad_(True) for i in range(3))
    pam = _rmask(s, w, times).expand(b, s, s).gather(dim=-1, index=pivot_idx.unsqueeze(1).expand(b, s, n_piv))
    torch.set_num_threads(max(1, min(16, os.cpu_count() or 1)))
    o = SD.sparse_attention(q, k, v, pivot_idx, pam, w, times, keep, P)
    o.backward(heads_first(d_out))
    o_tok = o.detach().permute(0, 2, 1, 3).reshape(b, s, h)
    err = (ctx.float().cpu() - o_tok).abs().max().item() / o_tok.abs().max().item()
    print("s=%d w=%d x%d piv=%d p=%.1f: fwd rel err %.3e" % (s, w, times, n_piv, P, err))
    assert err < 2e-2
    dq = dqkv.float().cpu()
    for name, got, ref in (("dq", dq[..., :h], q.grad), ("dk", dq[..., h:2 * h], k.grad), ("dv", dq[..., 2 * h:], v.grad)):
        ref_tok = ref.permute(0, 2, 1, 3).reshape(b, s, h)
        e = (got - ref_tok).abs().max().item() / ref_tok.abs().max().item()
        print("   %s rel err %.3e" % (name, e))
        assert e < 4e-2, (name, e)


def _corr(a, b):
    a, b = a.float(), b.float()
    a, b = a - a.mean(), b - b.mean()
    return ((a * b).mean() / (a.std() * b.std() + 1e-12)).item()


def test_sparse_dropout_mask_statistics():
    """Keep rate and independence at the CogView-sr shape (s = 4096, w = 128, times = 6, 768 pivots), separately over
    visible band entries and visible pivot entries; pivot slot t*128 + x and band key t*128 + x of the same query must be
    independent (disjoint counters); the bits are a pure function of (seed, site)."""
    from cogview_b200 import ops
    b, nh, s, w, times, n_piv = 1, 4, 4096, 128, 6, 768
    h = nh * 64
    g = torch.Generator(device="cuda").manual_seed(0)
    qkv = torch.randn((b, s, 3 * h), generator=g, device="cuda").bfloat16()
    pivot_idx = _pivots(b, s, n_piv, (100,), seed=5).cuda()

    def masks(site):
        _, m = ops.attn_sparse_fwd(qkv[..., :h], qkv[..., h:2 * h], qkv[..., 2 * h:], nh, pivot_idx, w, times,
                                   dropout=(P, 4321, site))
        return _decode(m, b, nh, s, n_piv, w, times)
    band_k, piv_k, band_q, piv_q, wb, wp = masks(3)
    band_vis, piv_vis = _visible(pivot_idx, s, w, times, "cuda")
    piv_vis = piv_vis[0]
    for what, keep, vis in (("band", band_k[0], band_vis), ("pivot", piv_k[0], piv_vis)):
        vals = keep[:, vis]
        n = vals.numel()
        rate = vals.float().mean().item()
        print("%s keep rate %.5f (expected %.5f, n = %d)" % (what, rate, 1 - P, n))
        assert abs(rate - (1 - P)) < 5 * (P * (1 - P) / n) ** 0.5
        k0 = keep[0]
        adj_k = vis[:, 1:] & vis[:, :-1]
        adj_q = vis[1:, :] & vis[:-1, :]
        c_key = _corr(k0[:, 1:][adj_k], k0[:, :-1][adj_k])
        c_qry = _corr(k0[1:, :][adj_q], k0[:-1, :][adj_q])
        c_head = _corr(keep[0][vis], keep[1][vis])
        print("  correlations: adjacent keys %.4f, adjacent queries %.4f, heads %.4f" % (c_key, c_qry, c_head))
        assert abs(c_key) < 5 / adj_k.sum().item() ** 0.5
        assert abs(c_qry) < 5 / adj_q.sum().item() ** 0.5
        assert abs(c_head) < 5 / vis.sum().item() ** 0.5
    # pivot slot x against band key x of the same query, wherever both tiles are in the query's list
    both = wb[:, :n_piv] & wp
    c_cross = _corr(piv_q[0][:, both], band_q[0][:, :, :n_piv][:, both])
    print("pivot slot vs band key of the same tile index: corr %.4f (n = %d)" % (c_cross, both.sum().item() * nh))
    assert both.sum().item() > 0 and abs(c_cross) < 5 / (both.sum().item() * nh) ** 0.5
    # pure function of (seed, site)
    again = masks(3)
    assert torch.equal(again[0] & band_vis, band_k & band_vis) and torch.equal(again[2] & wb, band_q & wb)
    assert torch.equal(again[3] & wp, piv_q & wp)
    other = masks(4)
    changed = (other[0][:, :, band_vis] != band_k[:, :, band_vis]).float().mean().item()
    print("other site: %.3f of the visible band bits differ" % changed)
    assert changed > 0.1


def _sparse_layer(h=256, heads=4, w=64, times=2, p_attn=P):
    from cogview_b200.mpu.sparse_transformer import GPT2ParallelTransformerLayer, unscaled_init_method
    torch.manual_seed(11)
    layer = GPT2ParallelTransformerLayer(h, heads, p_attn, 0.0, 1e-5, unscaled_init_method(0.02), query_window=w,
                                         key_window_times=times)
    with torch.no_grad():
        for n, prm in layer.named_parameters():
            if n.endswith("layernorm.weight"):
                prm.add_(0.1 * torch.randn_like(prm))
            elif n.endswith("bias"):
                prm.normal_(0.0, 0.02)
    return layer.cuda().bfloat16().train()


def test_layer_with_sparse_dropout_matches_oracle():
    from cogview_b200 import ops
    from cogview_b200.mpu.sparse_transformer import SparseSpec, layer_backward, layer_forward
    b, s, h, heads, w, times, n_piv = 2, 256, 256, 4, 64, 2, 48
    layer = _sparse_layer(h, heads, w, times)
    pivot_idx = _pivots(b, s, n_piv, (32, 32), seed=8)
    spec = SparseSpec(pivot_idx.cuda(), w, times)
    g = torch.Generator().manual_seed(12)
    x = torch.randn((b * s, h), generator=g)
    d_out = torch.randn((b * s, h), generator=g)
    P16 = tuple(prm.detach() for prm in layer.param_list())
    xc = x.cuda()
    drops = {'attn': (P, 999, 41), 'out': (0.0, 0, 0), 'mlp': (0.0, 0, 0)}
    save = []
    out, _ = layer_forward(xc, ops.absmax(xc), P16, heads, 1e-5, b, s, spec, save=save, drops=drops)
    mask = drops['attn_mask']
    d_x, grads = layer_backward(d_out.cuda(), save, P16, heads, b, s, spec, drops=drops)
    torch.cuda.synchronize()
    band_k, piv_k, _, _, _, _ = _decode(mask, b, heads, s, n_piv, w, times)
    keep = _to_reference_layout(band_k, piv_k, s, w, times).cpu()
    pre = 'transformer.layers.0.'
    sd = {pre + n: prm.detach().float().cpu().requires_grad_(True) for n, prm in layer.named_parameters()}
    xr = x.view(b, s, h).clone().requires_grad_(True)
    pam = _rmask(s, w, times).expand(b, s, s).gather(dim=-1, index=pivot_idx.unsqueeze(1).expand(b, s, n_piv))
    o = SD.transformer_layer(sd, 0, xr, pam, heads, pivot_idx, w, times, keep, P)
    o.backward(d_out.view(b, s, h))
    scale = o.abs().max().item()
    err = (out.float().cpu().view(b, s, h) - o.detach()).abs().max().item()
    print("layer with sparse dropout: out max|diff| %.3e (scale %.3e)" % (err, scale))
    assert err < 2e-2 * scale
    from cogview_b200.mpu.sparse_transformer import _PARAM_ORDER
    for name, got in zip(("x",) + _PARAM_ORDER, (d_x,) + tuple(grads)):
        ref = xr.grad.view(b * s, h) if name == "x" else sd[pre + name].grad
        e = ((got.float().cpu().view(ref.shape) - ref).abs().max() / ref.abs().max().clamp_min(1e-12)).item()
        assert e < 6e-2, (name, e)


def test_layer_checkpoint_recomputation_is_bitwise_identical():
    from cogview_b200 import ops
    from cogview_b200.mpu import random as mrandom
    from cogview_b200.mpu.sparse_transformer import SparseSpec, checkpoint
    b, s, h, heads, w, times, n_piv = 2, 256, 256, 4, 64, 2, 48
    layer = _sparse_layer(h, heads, w, times)
    spec = SparseSpec(_pivots(b, s, n_piv, (32, 32), seed=8).cuda(), w, times)
    g = torch.Generator().manual_seed(13)
    x0 = torch.randn((b * s, h), generator=g).cuda()
    d_out = torch.randn((b * s, h), generator=g).cuda()

    def run(use_ckpt, counter):
        mrandom.set_dropout_site_counter(counter)
        for prm in layer.parameters():
            prm.grad = None
        x = x0.clone().requires_grad_(True)
        am = ops.absmax(x0)
        if use_ckpt:
            out, _ = checkpoint(lambda x_, am_: layer.fused_forward(x_, am_, b, s, spec), x, am)
        else:
            out, _ = layer.fused_forward(x, am, b, s, spec)
        out.backward(d_out)
        return out.detach().clone(), [x.grad.clone()] + [prm.grad.clone() for prm in layer.param_list()]
    o0, g0 = run(False, 200)
    o1, g1 = run(True, 200)
    o2, _ = run(False, 600)
    assert torch.equal(o0, o1) and all(torch.equal(a, c) for a, c in zip(g0, g1))
    assert not torch.equal(o0, o2)


def _model(p):
    from cogview_b200.model import GPT2Model
    m = GPT2Model(num_layers=2, vocab_size=58240, hidden_size=256, num_attention_heads=4, embedding_dropout_prob=p,
                  attention_dropout_prob=p, output_dropout_prob=p, max_sequence_length=256, max_memory_length=0,
                  checkpoint_activations=True, checkpoint_num_layers=1, query_window=64, key_window_times=2,
                  num_pivot=48)
    m.load_state_dict(recipes.gpt2_state_dict(seed=21, num_layers=2, vocab_size=58240, hidden_size=256,
                                              num_attention_heads=4, max_sequence_length=256))
    return m.cuda().bfloat16()


def _model_inputs():
    s = 256
    tokens = recipes.text_image_tokens(2, 32, s - 32, seed=3)
    labels = torch.roll(tokens, -1, dims=1)
    pos = torch.arange(s).unsqueeze(0).expand(2, -1).contiguous()
    img = tokens < recipes.IMG_VOCAB
    return (tokens.cuda(), pos.cuda(), torch.tril(torch.ones((1, 1, s, s), device="cuda")), (~img).cuda(),
            img.cuda()), labels.cuda()


def test_model_sparse_training_with_dropout_is_reproducible():
    """2-layer GPT2Model, is_sparse = 1, checkpoint_activations, every dropout at 0.1: trains (this raised before),
    two runs with the same seeds and site counter are bitwise equal, another site counter gives another loss."""
    from cogview_b200 import mpu
    from cogview_b200.mpu import random as mrandom
    m = _model(P).train()
    args, labels = _model_inputs()

    def step(counter):
        torch.manual_seed(4321)
        random.seed(77)
        mrandom.set_dropout_site_counter(counter)
        m.zero_grad(set_to_none=True)
        logits, *_ = m(*args, 1)
        loss = mpu.vocab_parallel_cross_entropy(logits.contiguous().float(), labels).mean()
        loss.backward()
        return loss.item(), {n: prm.grad.float().clone() for n, prm in m.named_parameters()}
    l0, g0 = step(100)
    l1, g1 = step(100)
    l2, _ = step(500)
    print("sparse training step with dropout: loss %.5f (other sites %.5f)" % (l0, l2))
    assert l0 == l1 and all(torch.equal(g0[n], g1[n]) for n in g0)
    assert l2 != l0
    assert torch.isfinite(torch.tensor(l0)) and all(torch.isfinite(v).all() for v in g0.values())


def test_model_sparse_eval_ignores_dropout():
    ms = [_model(p).eval() for p in (P, 0.0)]
    args, _ = _model_inputs()
    outs = []
    for m in ms:
        random.seed(77)
        with torch.no_grad():
            logits, *_ = m(*args, 1)
        outs.append(logits)
    assert torch.equal(outs[0], outs[1])


def test_standalone_sparse_attention_with_dropout():
    from cogview_b200 import ops
    from cogview_b200.mpu.sparse_transformer import sparse_attention
    b, nh, s, hn, w, times, n_piv = 2, 3, 512, 64, 64, 3, 96
    gen = torch.Generator().manual_seed(31)
    q, k, v = (torch.randn((b, nh, s, hn), generator=gen).bfloat16() for _ in range(3))
    d_out = torch.randn((b, nh, s, hn), generator=gen)
    pivot_idx = _pivots(b, s, n_piv, (48, 20), seed=1234)
    qg, kg, vg = (t.cuda().requires_grad_(True) for t in (q, k, v))
    drop = torch.nn.Dropout(P).train()
    torch.manual_seed(5)
    out = sparse_attention(qg, kg, vg, pivot_idx.cuda(), None, w, times, attention_dropout=drop)
    out.float().backward(d_out.cuda())
    # the keep bits of that call: same (p, seed drawn from torch's generator, site 0)
    torch.manual_seed(5)
    seed = int(torch.randint(0, 2 ** 62, (1,)).item())

    def tok(t):
        return t.cuda().permute(0, 2, 1, 3).reshape(b, s, nh * hn).contiguous()
    ctx, mask = ops.attn_sparse_fwd(tok(q), tok(k), tok(v), nh, pivot_idx.cuda(), w, times, dropout=(P, seed, 0))
    assert torch.equal(ctx.view(b, s, nh, hn).permute(0, 2, 1, 3), out.detach())
    band_k, piv_k, _, _, _, _ = _decode(mask, b, nh, s, n_piv, w, times)
    keep = _to_reference_layout(band_k, piv_k, s, w, times).cpu()
    qr, kr, vr = (t.float().requires_grad_(True) for t in (q, k, v))
    pam = _rmask(s, w, times).expand(b, s, s).gather(dim=-1, index=pivot_idx.unsqueeze(1).expand(b, s, n_piv))
    o = SD.sparse_attention(qr, kr, vr, pivot_idx, pam, w, times, keep, P)
    o.backward(d_out)
    assert (out.float().cpu() - o.detach()).abs().max().item() < 2e-2 * o.abs().max().item()
    for name, got, ref in (("dq", qg.grad, qr.grad), ("dk", kg.grad, kr.grad), ("dv", vg.grad, vr.grad)):
        e = ((got.float().cpu() - ref).abs().max() / ref.abs().max()).item()
        assert e < 4e-2, (name, e)
    # eval mode: no dropout, bitwise the p = 0 result
    drop.eval()
    with torch.no_grad():
        a = sparse_attention(q.cuda(), k.cuda(), v.cuda(), pivot_idx.cuda(), None, w, times, attention_dropout=drop)
        z = sparse_attention(q.cuda(), k.cuda(), v.cuda(), pivot_idx.cuda(), None, w, times)
    assert torch.equal(a, z)
