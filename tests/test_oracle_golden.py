"""CPU: the travelling oracle (oracle/cogview_oracle.py) against the golden vectors produced by the
UNMODIFIED reference (oracle/make_golden.py).  This is the pin that makes the oracle trustworthy wherever
the reference itself is not available."""
import os

import numpy as np
import torch

from oracle import cogview_oracle as O
from oracle import recipes


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name), allow_pickle=False)


def test_weight_recipe_is_reproducible(golden_dir):
    g = _load(golden_dir, "gpt2_config1.npz")
    sd = recipes.gpt2_state_dict(**recipes.CONFIG1)
    chk = sum(float(v.double().sum()) for v in sd.values())
    assert abs(chk - float(g["weight_checksum"])) < 1e-6
    assert np.array_equal(recipes.text_image_tokens(2, 64, 65, seed=0).numpy(), g["tokens_full"])


def test_gpt2_forward_loss_backward_match_reference(golden_dir):
    g = _load(golden_dir, "gpt2_config1.npz")
    cfg = recipes.CONFIG1
    sd = {k: v.clone().requires_grad_(True) for k, v in recipes.gpt2_state_dict(**cfg).items()}
    tf = torch.from_numpy(g["tokens_full"])
    tokens, labels = tf[:, :-1].contiguous(), tf[:, 1:].contiguous()
    s = tokens.shape[1]
    pos = torch.arange(s).unsqueeze(0).expand_as(tokens)
    mask = torch.tril(torch.ones((1, 1, s, s)))
    logits, _ = O.gpt2_forward(sd, cfg["num_attention_heads"], tokens, pos, mask)
    stride = int(g["vocab_stride"])
    assert np.allclose(logits.detach()[:, :, ::stride].numpy(), g["logits_strided"], atol=2e-5)
    assert np.array_equal(logits.detach().argmax(-1).numpy(), g["logits_argmax"])          # bit-exact arg-max
    top8 = torch.topk(logits.detach(), 8, dim=-1)
    assert np.array_equal(top8.indices.numpy(), g["logits_top8_idx"])
    losses = O.vocab_parallel_cross_entropy(logits, labels)
    assert np.allclose(losses.detach().numpy(), g["losses"], atol=2e-5)
    loss = O.weighted_loss(losses, tokens, torch.ones_like(tokens, dtype=torch.float), recipes.IMG_VOCAB,
                           float(g["txt_loss_scale"]))
    assert abs(loss.item() - float(g["loss"])) < 1e-5
    loss.backward()
    names = [str(n) for n in g["grad_names"]]
    for i, n in enumerate(names):
        gr = sd[n].grad.reshape(-1)
        idx = torch.linspace(0, gr.numel() - 1, 64).long()
        assert np.allclose(gr[idx].numpy(), g["grad_samples"][i], atol=2e-6), n
        assert abs(float(gr.norm()) - g["grad_norms"][i]) <= 1e-4 * max(1.0, g["grad_norms"][i]), n
    # int `sep` mask form
    lg, _ = O.gpt2_forward({k: v.detach() for k, v in sd.items()}, cfg["num_attention_heads"], tokens, pos, 40)
    assert np.allclose(lg[:, :, ::int(g["sep40_vocab_stride"])].numpy(), g["logits_sep40_strided"], atol=2e-5)


def test_gpt2_decode_with_mems_matches_reference(golden_dir):
    g = _load(golden_dir, "gpt2_config1.npz")
    cfg = recipes.CONFIG1
    sd = recipes.gpt2_state_dict(**cfg)
    tf = torch.from_numpy(g["tokens_full"])
    ctx = tf[:, :64]
    pos = torch.arange(64).unsqueeze(0).expand(2, -1)
    with torch.no_grad():
        lg, mems = O.gpt2_forward(sd, cfg["num_attention_heads"], ctx, pos, torch.tril(torch.ones((1, 1, 64, 64))),
                                  max_memory_length=128)
        toks = []
        for t in range(64, 128):
            nxt = lg[:, -1, :recipes.IMG_VOCAB].argmax(-1)
            toks.append(nxt)
            lg, mems = O.gpt2_forward(sd, cfg["num_attention_heads"], nxt.unsqueeze(1),
                                      torch.full((2, 1), t, dtype=torch.long), 0, mems=mems, max_memory_length=128)
    assert np.array_equal(torch.stack(toks, 1).numpy(), g["decode_tokens"])               # bit-exact tokens
    assert np.allclose(lg[:, -1, ::int(g["vocab_stride"])].numpy(), g["decode_last_logits_strided"], atol=2e-5)


def _attention_inputs(g):
    b, nh, s, hn, w, times, n_piv, sq = [int(x) for x in g["dims"]]
    gen = torch.Generator().manual_seed(int(g["seed"]))
    q, k, v = (torch.randn((b, nh, s, hn), generator=gen) for _ in range(3))
    pivot_idx = torch.from_numpy(g["pivot_idx"])
    gcount = s // w
    tmp = torch.ones((gcount - times + 1, w, w))
    tmp = torch.tril(1 - torch.block_diag(*tmp))
    rmask = torch.nn.functional.pad(tmp, (0, (times - 1) * w, (times - 1) * w, 0))
    pam = rmask.expand(b, s, s).gather(dim=-1, index=pivot_idx.unsqueeze(1).expand(b, s, n_piv))
    return q, k, v, pivot_idx, pam, (b, nh, s, hn, w, times, n_piv, sq)


def test_attention_variants_match_reference(golden_dir):
    g = _load(golden_dir, "attention.npz")
    q, k, v, pivot_idx, pam, (b, nh, s, hn, w, times, n_piv, sq) = _attention_inputs(g)
    dense = O.standard_attention(q, k, v, torch.tril(torch.ones((1, 1, s, s))))
    assert np.allclose(dense.numpy()[:, :, ::7], g["dense"], atol=1e-5)
    sp = O.sparse_attention(q, k, v, pivot_idx, pam, w, times)
    assert np.allclose(sp.numpy()[:, :, ::7], g["sparse_train"], atol=1e-5)
    pw = torch.cat((pivot_idx, torch.arange(s - times * w, s).expand(b, -1)), dim=-1)
    inf = O.sparse_attention_inference(q[:, :, -sq:], k, v, pw)
    assert np.allclose(inf.numpy(), g["sparse_infer"], atol=1e-5)


def test_vqvae_matches_reference(golden_dir):
    g = _load(golden_dir, "vqvae_64.npz")
    sd = recipes.vqvae_state_dict(seed=0)
    img = recipes.images(2, size=64, seed=0)
    with torch.no_grad():
        z = O.vq_encoder(sd, img)
    assert np.allclose(z.numpy(), g["z"], atol=2e-5)
    codes = O.img2code(sd, img)
    assert np.array_equal(codes.numpy(), g["codes"])                                      # bit-exact indices
    rec = O.code2img(sd, codes.view(2, 8, 8))
    assert np.allclose(rec.numpy(), g["recon"], atol=2e-5)


def test_sparse_training_attention_two_pass_decomposition(golden_dir):
    """Row a7 (not yet built in CUDA): the band + pivot two-pass form with a joint log-sum-exp that a tile-scheduled
    kernel would run (oracle/sparse_decomposition.py) reproduces the reference's sparse_attention — forward against
    the golden output, visibility rules against the reference's rmask, backward against autograd."""
    from oracle import sparse_decomposition as SD
    g = _load(golden_dir, "attention.npz")
    q, k, v, pivot_idx, pam, (b, nh, s, hn, w, times, n_piv, sq) = _attention_inputs(g)
    band, piv = SD.visibility(s, pivot_idx, w, times)
    assert torch.equal(piv.float(), pam)                                   # closed form == gathered rmask
    wm = torch.tril(torch.ones(s, s)) * (1 - torch.nn.functional.pad(
        torch.tril(1 - torch.block_diag(*torch.ones((s // w - times + 1, w, w)))), (0, (times - 1) * w, (times - 1) * w, 0)))
    assert torch.equal(band.float(), wm)                                   # band == causal minus the pivot region
    out, lse = SD.sparse_attention_two_pass(q, k, v, pivot_idx, w, times)
    assert np.allclose(out.numpy()[:, :, ::7], g["sparse_train"], atol=1e-5)
    qr, kr, vr = (t.clone().requires_grad_(True) for t in (q, k, v))
    ref = O.sparse_attention(qr, kr, vr, pivot_idx, pam, w, times)
    gen = torch.Generator().manual_seed(11)
    d_out = torch.randn(ref.shape, generator=gen)
    ref.backward(d_out)
    dq, dk, dv = SD.sparse_attention_two_pass_backward(q, k, v, pivot_idx, w, times, out, lse, d_out)
    for got, want in ((dq, qr.grad), (dk, kr.grad), (dv, vr.grad)):
        assert (got - want).abs().max().item() < 2e-5 * max(1.0, want.abs().max().item())
