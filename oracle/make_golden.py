"""TEST INFRASTRUCTURE — golden-vector generator.  Runs ONLY in the build container.

  python oracle/make_golden.py

1. Places the UNMODIFIED reference under oracle/_ref (oracle/build_ref.py), imports it (oracle/ref_harness.py) and runs it on the seeded inputs of
   oracle/recipes.py (SURVEY §8(d) config 1; VQ-VAE new_model()).
2. Asserts the travelling restatement oracle/cogview_oracle.py reproduces the reference (fp32).
3. Writes compact fixtures to tests/golden/ (outputs only — weights/inputs are regenerated from seeds).
"""
import os
import random
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import cogview_oracle as O  # noqa: E402
from oracle import build_ref, recipes, ref_harness  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
VOCAB_STRIDE = 97  # logits are stored on every 97th vocab column (+ arg-max / top-8 per position)
SEP40_VOCAB_STRIDE = 8 * VOCAB_STRIDE  # the int-sep logits on a coarser sample keep gpt2_config1.npz under 1 MB


def close(a, b, tol, what):
    err = (a - b).abs().max().item()
    scale = b.abs().max().item()
    print("  %-46s max|diff| %.3e (scale %.3e)" % (what, err, scale))
    assert err <= tol * max(1.0, scale), what
    return err


def sample_grad(g):
    flat = g.reshape(-1)
    idx = torch.linspace(0, flat.numel() - 1, 64).long()
    return flat[idx].numpy(), float(flat.norm())


def gpt2_golden(ref):
    cfg = recipes.CONFIG1
    sd = recipes.gpt2_state_dict(**cfg)
    tokens_full = recipes.text_image_tokens(2, 64, 65, seed=0)       # 129 tokens -> 128 inputs / labels
    tokens, labels = tokens_full[:, :-1].contiguous(), tokens_full[:, 1:].contiguous()
    s = tokens.shape[1]
    pos = torch.arange(s).unsqueeze(0).expand_as(tokens)
    mask = torch.tril(torch.ones((1, 1, s, s)))

    def make_ref(max_mem):
        m = ref["gpt2_modeling"].GPT2Model(
            num_layers=cfg["num_layers"], vocab_size=cfg["vocab_size"], hidden_size=cfg["hidden_size"],
            num_attention_heads=cfg["num_attention_heads"], embedding_dropout_prob=0.0, attention_dropout_prob=0.0,
            output_dropout_prob=0.0, max_sequence_length=cfg["max_sequence_length"], max_memory_length=max_mem,
            checkpoint_activations=False)
        m.load_state_dict(sd)
        return m

    # ---- training forward / loss / backward through the reference ----
    model = make_ref(0)
    logits, *_ = model(tokens, pos, mask, None, None, 0)
    losses = ref["mpu"].vocab_parallel_cross_entropy(logits.contiguous().float(), labels)
    loss_mask = torch.ones_like(tokens, dtype=torch.float)
    txt_scale = 2.5
    lm = loss_mask.clone()
    lm[(tokens >= recipes.IMG_VOCAB)] *= txt_scale           # pretrain_gpt2.py:300-314
    loss = torch.sum(losses.view(-1) * lm.view(-1)) / lm.sum()
    loss.backward()
    ref_grads = {k: p.grad.detach().clone() for k, p in model.named_parameters()}

    # ---- the restatement must reproduce it ----
    print("GPT-2 config 1: restatement vs reference")
    sdr = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    o_logits, _ = O.gpt2_forward(sdr, cfg["num_attention_heads"], tokens, pos, mask)
    o_losses = O.vocab_parallel_cross_entropy(o_logits, labels)
    o_loss = O.weighted_loss(o_losses, tokens, loss_mask, recipes.IMG_VOCAB, txt_scale)
    o_loss.backward()
    close(o_logits.detach(), logits.detach(), 2e-5, "logits")
    close(o_losses.detach(), losses.detach(), 2e-5, "per-token loss")
    close(o_loss.detach(), loss.detach(), 1e-6, "weighted loss")
    for k in ref_grads:
        close(sdr[k].grad, ref_grads[k], 2e-5, "grad " + k)
    # int-sep mask form (mpu/sparse_transformer.py:477-489)
    lg_sep, *_ = model(tokens, pos, 40, None, None, 0)
    o_sep, _ = O.gpt2_forward(sd, cfg["num_attention_heads"], tokens, pos, 40)
    close(o_sep, lg_sep.detach(), 2e-5, "logits with int sep=40")

    # ---- decode with hidden-state mems: prefill 64, then 64 greedy steps (generation/sampling.py:126-151) ----
    model_m = make_ref(cfg["max_sequence_length"])
    model_m.eval()
    with torch.no_grad():
        ctx = tokens[:, :64]
        lg, *mems = model_m(ctx, pos[:, :64], torch.tril(torch.ones((1, 1, 64, 64))), None, None, 0)
        o_lg, o_mems = O.gpt2_forward(sd, cfg["num_attention_heads"], ctx, pos[:, :64],
                                      torch.tril(torch.ones((1, 1, 64, 64))), max_memory_length=128)
        gen, step_logit_samples = [], []
        cur = ctx
        for t in range(64, 128):
            nxt = lg[:, -1, :recipes.IMG_VOCAB].argmax(-1)      # image tokens only, like invalid_slices
            o_nxt = o_lg[:, -1, :recipes.IMG_VOCAB].argmax(-1)
            assert torch.equal(nxt, o_nxt), "greedy token mismatch at step %d" % t
            gen.append(nxt)
            step_logit_samples.append(lg[:, -1, ::VOCAB_STRIDE].clone())
            p = torch.full((2, 1), t, dtype=torch.long)
            lg, *mems = model_m(nxt.unsqueeze(1), p, 0, None, None, 0, *mems)
            o_lg, o_mems = O.gpt2_forward(sd, cfg["num_attention_heads"], nxt.unsqueeze(1), p, 0, mems=o_mems,
                                          max_memory_length=128)
        close(o_lg, lg, 2e-5, "decode: last-step logits")
        gen = torch.stack(gen, 1)

    top8 = torch.topk(logits.detach(), 8, dim=-1)
    np.savez_compressed(
        os.path.join(GOLD, "gpt2_config1.npz"),
        tokens_full=tokens_full.numpy(), txt_loss_scale=np.float32(txt_scale),
        weight_checksum=np.float64(sum(float(v.double().sum()) for v in sd.values())),
        logits_strided=logits.detach()[:, :, ::VOCAB_STRIDE].numpy(), vocab_stride=np.int64(VOCAB_STRIDE),
        logits_argmax=logits.detach().argmax(-1).numpy(),
        logits_top8_val=top8.values.numpy(), logits_top8_idx=top8.indices.numpy(),
        losses=losses.detach().numpy(), loss=np.float32(loss.item()),
        logits_sep40_strided=lg_sep.detach()[:, :, ::SEP40_VOCAB_STRIDE].numpy(),
        sep40_vocab_stride=np.int64(SEP40_VOCAB_STRIDE),
        grad_names=np.array(list(ref_grads.keys())),
        grad_samples=np.stack([sample_grad(g)[0] for g in ref_grads.values()]),
        grad_norms=np.array([sample_grad(g)[1] for g in ref_grads.values()], dtype=np.float64),
        decode_tokens=gen.numpy(), decode_step_logits=torch.stack(step_logit_samples, 1).numpy(),
        decode_last_logits_strided=lg[:, -1, ::VOCAB_STRIDE].numpy(),
    )


def attention_golden(ref):
    """Function-level fixtures for the three attention variants (mpu/sparse_transformer.py:652-750), with the
    mask recipe of the in-file test_sparse_attention (:753-784) at reduced size."""
    st = ref["sparse_transformer"]
    print("attention functions: restatement vs reference")
    g = torch.Generator().manual_seed(7)
    b, nh, hn = 2, 3, 64
    s, w, times, n_piv = 512, 64, 3, 96
    q, k, v = (torch.randn((b, nh, s, hn), generator=g) for _ in range(3))
    # dense, causal
    mask = torch.tril(torch.ones((1, 1, s, s)))
    r_dense = st.standard_attention(q, k, v, mask)
    close(O.standard_attention(q, k, v, mask), r_dense, 1e-5, "standard_attention (causal)")
    # sparse training
    random.seed(1234)
    txt_n = [48, 20]
    pivot_idx = torch.stack([
        torch.cat((torch.arange(0, txt_n[i]),
                   torch.tensor(random.sample(range(txt_n[i], s), n_piv - txt_n[i]), dtype=torch.long)))
        for i in range(b)])
    gcount = s // w
    tmp = torch.ones((gcount - times + 1, w, w))
    tmp = torch.tril(1 - torch.block_diag(*tmp))
    rmask = torch.nn.functional.pad(tmp, (0, (times - 1) * w, (times - 1) * w, 0))
    pam = rmask.expand(b, s, s).gather(dim=-1, index=pivot_idx.unsqueeze(1).expand(b, s, n_piv))
    r_sparse = st.sparse_attention(q, k, v, pivot_idx, pam, w, times, None)
    close(O.sparse_attention(q, k, v, pivot_idx, pam, w, times), r_sparse, 1e-5, "sparse_attention (train)")
    # sparse inference: last 5 queries, keys = pivots U last window
    sq = 5
    pw_idx = torch.cat((pivot_idx[:, :n_piv], torch.arange(s - times * w, s).expand(b, -1)), dim=-1)
    r_inf = st.sparse_attention_inference(q[:, :, -sq:], k, v, pw_idx)
    close(O.sparse_attention_inference(q[:, :, -sq:], k, v, pw_idx), r_inf, 1e-5, "sparse_attention_inference")
    np.savez_compressed(os.path.join(GOLD, "attention.npz"), seed=np.int64(7),
                        dims=np.array([b, nh, s, hn, w, times, n_piv, sq]), pivot_idx=pivot_idx.numpy(),
                        dense=r_dense.numpy().astype(np.float32)[:, :, ::7],
                        sparse_train=r_sparse.numpy()[:, :, ::7], sparse_infer=r_inf.numpy())


def vqvae_golden(ref):
    print("VQ-VAE: restatement vs reference")
    sd = recipes.vqvae_state_dict(seed=0)
    model = ref["vq_api"].new_model()
    missing = model.load_state_dict(sd)
    model.eval()
    img = recipes.images(2, size=64, seed=0)
    with torch.no_grad():
        z_ref = model.enc_b(img)
        codes = ref["vq_api"].img2code(model, img)
        rec = ref["vq_api"].code2img(model, codes.view(2, 8, 8))
        z = O.vq_encoder(sd, img)
        close(z, z_ref, 2e-5, "encoder output z")
        o_codes = O.img2code(sd, img)
        assert torch.equal(o_codes, codes), "codes differ"
        print("  codes bit-exact: True")
        close(O.code2img(sd, codes.view(2, 8, 8)), rec, 2e-5, "decoded image")
        d = O.vq_distances(z_ref.reshape(-1, 256), sd['quantize_t.embed'])
        top2 = torch.topk(-d, 2, dim=1).values
        gap = (top2[:, 0] - top2[:, 1])
        print("  nearest/second-nearest distance gap: min %.3e median %.3e" % (gap.min(), gap.median()))
    np.savez_compressed(os.path.join(GOLD, "vqvae_64.npz"), z=z_ref.numpy(), codes=codes.numpy(),
                        recon=rec.numpy(), min_gap=np.float32(gap.min().item()))


def vqvae_golden_256(ref, n=17):
    """configs[3] shapes: 256x256 images, 512-channel maps, 32x32 codes, more images than one batch chunk (16).
    Stored: codes, the reference's nearest / second-nearest distance gap per code (which codes are decisive for a
    bf16 encoder), strided samples of z and of the reconstruction."""
    print("VQ-VAE 256x256: reference outputs for %d images" % n)
    sd = recipes.vqvae_state_dict(seed=0)
    model = ref["vq_api"].new_model()
    model.load_state_dict(sd)
    model.eval()
    img = recipes.images(n, size=256, seed=5)
    with torch.no_grad():
        z_ref = model.enc_b(img)                                   # [n, 32, 32, 256]
        codes = ref["vq_api"].img2code(model, img)                 # [n, 1024]
        rec = ref["vq_api"].code2img(model, codes.view(n, 32, 32))
        o_codes = O.img2code(sd, img)
        assert torch.equal(o_codes, codes), "oracle codes differ from the reference at 256x256"
        close(O.code2img(sd, codes.view(n, 32, 32)), rec, 2e-5, "decoded 256x256 image")
        d = O.vq_distances(z_ref.reshape(-1, 256), sd['quantize_t.embed'])
        top2 = torch.topk(-d, 2, dim=1).values
        gap = (top2[:, 0] - top2[:, 1]).view(n, 1024)
    print("  gap: min %.3e median %.3e; z scale %.3f" % (gap.min(), gap.median(), z_ref.abs().max()))
    np.savez_compressed(os.path.join(GOLD, "vqvae_256.npz"), codes=codes.numpy().astype(np.int16),
                        gap=gap.numpy().astype(np.float32), z_strided=z_ref[:, ::8, ::8, :].numpy(),
                        z_absmax=np.float32(z_ref.abs().max().item()),
                        recon_strided=rec[:, :, ::16, ::16].numpy(), recon_absmax=np.float32(rec.abs().max().item()))


def main():
    os.makedirs(GOLD, exist_ok=True)
    torch.set_num_threads(8)
    if not build_ref.build():
        raise SystemExit("make_golden: the reference is not available under oracle/_ref")
    ref = ref_harness.load()
    gpt2_golden(ref)
    attention_golden(ref)
    vqvae_golden(ref)
    vqvae_golden_256(ref)
    print("golden fixtures written to", GOLD)


if __name__ == "__main__":
    main()
