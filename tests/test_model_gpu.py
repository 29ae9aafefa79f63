"""GPU parity of the drop-in GPT2Model (cogview_b200.model) against the CPU oracle and the golden vectors
produced by the unmodified reference (SURVEY §8(d) config 1: 2 layers, d=256, 4 heads, V=58240, 128 tokens).

Tolerances (bf16 tensor-core math vs the fp32 oracle): logits within 2e-2 of the logit scale, per-token loss
within 1e-2 absolute... stated per assertion below.  Arg-max: must agree wherever the oracle's top-1/top-2
margin exceeds the logit tolerance, and the overall agreement is reported."""
import os

import numpy as np
import pytest
import torch

from oracle import cogview_oracle as O
from oracle import recipes

pytestmark = pytest.mark.gpu

CFG = recipes.CONFIG1


def build(max_memory_length=0, mems_mode=None, checkpoint_activations=False):
    from cogview_b200.model import GPT2Model
    m = GPT2Model(num_layers=CFG["num_layers"], vocab_size=CFG["vocab_size"], hidden_size=CFG["hidden_size"],
                  num_attention_heads=CFG["num_attention_heads"], embedding_dropout_prob=0.0,
                  attention_dropout_prob=0.0, output_dropout_prob=0.0,
                  max_sequence_length=CFG["max_sequence_length"], max_memory_length=max_memory_length,
                  checkpoint_activations=checkpoint_activations)
    m.load_state_dict(recipes.gpt2_state_dict(**CFG))
    m = m.cuda().bfloat16()
    if mems_mode:
        m.transformer.mems_mode = mems_mode
    return m


@pytest.fixture(scope="module")
def data(golden_dir):
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    g = np.load(os.path.join(golden_dir, "gpt2_config1.npz"))
    tf = torch.from_numpy(g["tokens_full"])
    tokens, labels = tf[:, :-1].contiguous(), tf[:, 1:].contiguous()
    s = tokens.shape[1]
    pos = torch.arange(s).unsqueeze(0).expand_as(tokens).contiguous()
    # the oracle runs on the bf16-rounded weights the GPU model holds, so only compute precision differs
    sd = {k: v.to(torch.bfloat16).float() for k, v in recipes.gpt2_state_dict(**CFG).items()}
    return dict(g=g, tokens=tokens, labels=labels, pos=pos, sd=sd, s=s)


def test_forward_logits_match_oracle_and_golden(data):
    m = build().eval()
    s = data["s"]
    mask = torch.tril(torch.ones((1, 1, s, s), device="cuda"))
    with torch.no_grad():
        logits, *mems = m(data["tokens"].cuda(), data["pos"].cuda(), mask, None, None, 0)
    assert mems == []
    lg = logits.float().cpu()
    o_logits, _ = O.gpt2_forward(data["sd"], CFG["num_attention_heads"], data["tokens"], data["pos"],
                                 torch.tril(torch.ones((1, 1, s, s))))
    scale = o_logits.abs().max().item()
    err = (lg - o_logits).abs().max().item()
    print("logits: max|diff| %.3e, scale %.3e" % (err, scale))
    assert err < 2e-2 * scale
    # against the reference's own (fp32-weight) outputs: strided logits within the same tolerance
    g = data["g"]
    stride = int(g["vocab_stride"])
    assert np.abs(lg[:, :, ::stride].numpy() - g["logits_strided"]).max() < 3e-2 * scale
    # arg-max: exact wherever the reference's top-2 margin exceeds the tolerance
    margin = torch.from_numpy(g["logits_top8_val"][..., 0] - g["logits_top8_val"][..., 1])
    am = lg.argmax(-1)
    ref_am = torch.from_numpy(g["logits_argmax"])
    decisive = margin > 2 * 2e-2 * scale
    assert torch.equal(am[decisive], ref_am[decisive])
    print("arg-max agreement with the reference: %d / %d (decisive positions: %d)" % (
        (am == ref_am).sum().item(), am.numel(), decisive.sum().item()))
    assert (am == ref_am).float().mean().item() > 0.97


def test_int_sep_mask_form(data):
    m = build().eval()
    with torch.no_grad():
        logits, *_ = m(data["tokens"].cuda(), data["pos"].cuda(), 40, None, None, 0)
    g = data["g"]
    stride = int(g["sep40_vocab_stride"])
    scale = np.abs(g["logits_sep40_strided"]).max()
    assert np.abs(logits.float().cpu()[:, :, ::stride].numpy() - g["logits_sep40_strided"]).max() < 3e-2 * scale


@pytest.mark.parametrize("mode", ["hidden", "kv"])
def test_decode_with_mems(data, mode):
    """prefill 64 tokens, then 64 greedy steps over the image vocabulary (generation/sampling.py:126-183)."""
    m = build(max_memory_length=CFG["max_sequence_length"], mems_mode=mode).eval()
    g = data["g"]
    ctx = data["tokens"][:, :64].cuda()
    pos = data["pos"][:, :64].cuda()
    ref_tokens = torch.from_numpy(g["decode_tokens"])          # [2, 64] greedy tokens of the reference
    stride = int(g["vocab_stride"])
    with torch.no_grad():
        lg, *mems = m(ctx, pos, torch.tril(torch.ones((1, 1, 64, 64), device="cuda")), None, None, 0)
        assert len(mems) == CFG["num_layers"] + 1 and mems[0].size(1) == 64
        agree, worst = 0, 0.0
        for i, t in enumerate(range(64, 128)):
            step_ref = torch.from_numpy(g["decode_step_logits"][:, i])          # logits that chose token t
            worst = max(worst, (lg[:, -1].float().cpu()[:, ::stride] - step_ref).abs().max().item())
            nxt = lg[:, -1, :recipes.IMG_VOCAB].float().argmax(-1).cpu()
            agree += int((nxt == ref_tokens[:, i]).sum())
            # teacher-force the reference's token so one near-tie does not derail the rest of the comparison
            feed = ref_tokens[:, i].cuda().unsqueeze(1)
            lg, *mems = m(feed, torch.full((2, 1), t, dtype=torch.long, device="cuda"), 0, None, None, 0, *mems)
            assert mems[0].size(1) == t + 1
        last = lg[:, -1].float().cpu()[:, ::stride].numpy()
    scale = np.abs(g["decode_last_logits_strided"]).max()
    print("[%s] decode: worst step-logit diff %.3e (scale %.3e); greedy agreement %d/128" % (mode, worst, scale, agree))
    assert worst < 3e-2 * scale
    assert np.abs(last - g["decode_last_logits_strided"]).max() < 3e-2 * scale
    assert agree >= 120


def test_state_dict_keys_match_reference_layout():
    m = build()
    keys = set(m.state_dict().keys())
    assert keys == set(recipes.gpt2_state_dict(**CFG).keys())
    from cogview_b200 import mpu
    assert all(getattr(p, "model_parallel", False) for n, p in m.named_parameters()
               if n.endswith("query_key_value.weight") or n == "word_embeddings.weight")
    assert isinstance(m.transformer.final_layernorm, mpu.LayerNorm)


@pytest.mark.parametrize("ckpt", [False, True])
def test_training_step_loss_and_grads(data, ckpt):
    """forward + mpu.vocab_parallel_cross_entropy + the reference's loss weighting (pretrain_gpt2.py:305-321) +
    backward; gradients against the oracle's autograd on the same (bf16-rounded) weights and against the
    reference's own gradient norms from the golden file."""
    from cogview_b200 import mpu
    m = build(checkpoint_activations=ckpt).train()
    g = data["g"]
    s = data["s"]
    tokens, labels = data["tokens"].cuda(), data["labels"].cuda()
    mask = torch.tril(torch.ones((1, 1, s, s), device="cuda"))
    logits, *_ = m(tokens, data["pos"].cuda(), mask, None, None, 0)
    losses = mpu.vocab_parallel_cross_entropy(logits.contiguous().float(), labels)
    txt_scale = float(g["txt_loss_scale"])
    lm = torch.ones_like(tokens, dtype=torch.float)
    lm[tokens >= recipes.IMG_VOCAB] *= txt_scale
    loss = torch.sum(losses.view(-1) * lm.view(-1)) / lm.sum()
    loss.backward()
    # oracle on the same weights
    sdr = {k: v.clone().requires_grad_(True) for k, v in data["sd"].items()}
    o_logits, _ = O.gpt2_forward(sdr, CFG["num_attention_heads"], data["tokens"], data["pos"],
                                 torch.tril(torch.ones((1, 1, s, s))))
    o_losses = O.vocab_parallel_cross_entropy(o_logits, data["labels"])
    o_loss = O.weighted_loss(o_losses, data["tokens"], torch.ones_like(data["tokens"], dtype=torch.float),
                             recipes.IMG_VOCAB, txt_scale)
    o_loss.backward()
    print("loss %.5f oracle %.5f reference %.5f" % (loss.item(), o_loss.item(), float(g["loss"])))
    assert (losses.float().cpu() - o_losses.detach()).abs().max().item() < 5e-2
    assert abs(loss.item() - o_loss.item()) < 1e-2
    assert abs(loss.item() - float(g["loss"])) < 2e-2
    names = [str(n) for n in g["grad_names"]]
    worst = ("", 0.0)
    for n, p in m.named_parameters():
        assert p.grad is not None, n
        ref = sdr[n].grad
        e = ((p.grad.float().cpu() - ref).abs().max() / ref.abs().max().clamp_min(1e-12)).item()
        if e > worst[1]:
            worst = (n, e)
        assert e < 6e-2, (n, e)
        gn = float(p.grad.float().norm())
        rn = float(g["grad_norms"][names.index(n)])
        assert abs(gn - rn) < 5e-2 * rn, (n, gn, rn)
    print("worst relative gradient error: %s %.3e" % worst)


def test_sparse_inference_equals_dense_when_window_covers_everything(data):
    """is_sparse=2 (mpu/sparse_transformer.py:498-520, 727-750): with key_length <= query_window * key_window_times the
    gathered key set is every key, so sparse decode must reproduce the dense KV-cache decode."""
    m = build(max_memory_length=CFG["max_sequence_length"], mems_mode="kv").eval()
    ctx = data["tokens"][:, :64].cuda()
    pos = data["pos"][:, :64].cuda()
    with torch.no_grad():
        img = ctx < recipes.IMG_VOCAB
        lg_s, *mems_s = m(ctx, pos, torch.tril(torch.ones((1, 1, 64, 64), device="cuda")), ~img, img, 2)
        lg_d, *mems_d = build(max_memory_length=CFG["max_sequence_length"], mems_mode="kv").eval()(
            ctx, pos, torch.tril(torch.ones((1, 1, 64, 64), device="cuda")), None, None, 0)
        scale = lg_d.abs().max().item()
        assert (lg_s - lg_d).abs().max().item() < 2e-2 * scale
        toks = ctx
        for t in range(64, 68):
            nxt = lg_s[:, -1, :recipes.IMG_VOCAB].float().argmax(-1, keepdim=True)
            toks = torch.cat((toks, nxt), dim=1)
            img = toks < recipes.IMG_VOCAB
            p = torch.full((2, 1), t, dtype=torch.long, device="cuda")
            lg_s, *mems_s = m(nxt, p, 0, ~img, img, 2, *mems_s)
        assert mems_s[0].size(1) == 68 and bool(torch.isfinite(lg_s).all())


def _fill(monkeypatch, graph_sampling, top_k, seed):
    """filling_sequence (generation/sampling.py:64-186) on the tiny model: 20 context tokens, 44 generated, 3 beams."""
    from cogview_b200.generation import sampling
    monkeypatch.setenv("COGVIEW_B200_GRAPH_SAMPLING", "1" if graph_sampling else "0")
    m = build(max_memory_length=CFG["max_sequence_length"], mems_mode="kv").eval()

    class A:
        temperature, top_p, is_sparse = 1.0, 0.0, 0
        img_tokenizer_num_tokens = recipes.IMG_VOCAB
    A.top_k = top_k

    tok = sampling.get_tokenizer(A)
    g = torch.Generator().manual_seed(3)
    text = torch.randint(recipes.IMG_VOCAB, recipes.IMG_VOCAB + 100, (18,), generator=g).tolist()
    seq = [tok['[ROI1]']] + text + [tok['[BASE]'], tok['[BOI1]']] + [-3] * 44
    torch.manual_seed(seed)
    with torch.no_grad():
        out = sampling.filling_sequence(m, torch.tensor(seq, dtype=torch.long, device="cuda"), A)
    return out.cpu(), len(seq)


def test_filling_sequence_graph_sampling_matches_eager_loop(monkeypatch):
    """The generation run with the sampling tail inside the decode graph (mpu/decode.py sample_run) against the
    per-token host loop: identical tokens for top-k = 1 (no randomness left), valid image codes for top-k = 200."""
    eager, n = _fill(monkeypatch, False, 1, 0)
    fused, _ = _fill(monkeypatch, True, 1, 0)
    assert eager.shape == fused.shape == (3, n)
    assert torch.equal(eager[:, :21], fused[:, :21])
    agree = (eager == fused).float().mean().item()
    assert agree == 1.0, agree
    sampled, _ = _fill(monkeypatch, True, 200, 1)
    assert sampled.shape == (3, n) and int(sampled[:, 21:].min()) >= 0 and int(sampled[:, 21:].max()) < recipes.IMG_VOCAB
    assert len({tuple(r.tolist()) for r in sampled[:, 21:]}) > 1          # beams diverge


def test_4b_shaped_layer_forward_backward_matches_oracle():
    """One CogView-base layer at its BASELINE shape (h = 2560, 40 heads, s = 1088 tokens, b = 1) through GPT2Model:
    logits, loss and every gradient against the fp32 oracle on the same (bf16-rounded) weights.  The vocabulary is cut
    to 2048 rows so that the CPU oracle finishes in seconds; every other dimension is the 4B model's."""
    from cogview_b200 import mpu
    from cogview_b200.model import GPT2Model
    cfg = dict(num_layers=1, vocab_size=2048, hidden_size=2560, num_attention_heads=40, max_sequence_length=1088)
    s = 1088
    sd32 = recipes.gpt2_state_dict(seed=11, **cfg)
    m = GPT2Model(num_layers=1, vocab_size=cfg["vocab_size"], hidden_size=cfg["hidden_size"],
                  num_attention_heads=cfg["num_attention_heads"], embedding_dropout_prob=0.0,
                  attention_dropout_prob=0.0, output_dropout_prob=0.0, max_sequence_length=s, max_memory_length=0,
                  checkpoint_activations=False)
    m.load_state_dict(sd32)
    m = m.cuda().bfloat16().train()
    g = torch.Generator().manual_seed(5)
    tokens = torch.randint(0, cfg["vocab_size"], (1, s), generator=g)
    labels = torch.randint(0, cfg["vocab_size"], (1, s), generator=g)
    pos = torch.arange(s).unsqueeze(0)
    logits, *_ = m(tokens.cuda(), pos.cuda(), torch.tril(torch.ones((1, 1, s, s), device="cuda")), None, None, 0)
    losses = mpu.vocab_parallel_cross_entropy(logits.contiguous().float(), labels.cuda())
    loss = losses.mean()
    loss.backward()
    sdr = {k: v.to(torch.bfloat16).float().requires_grad_(True) for k, v in sd32.items()}
    torch.set_num_threads(max(1, min(16, os.cpu_count() or 1)))
    o_logits, _ = O.gpt2_forward(sdr, cfg["num_attention_heads"], tokens, pos, torch.tril(torch.ones((1, 1, s, s))))
    o_losses = O.vocab_parallel_cross_entropy(o_logits, labels)
    o_loss = o_losses.mean()
    o_loss.backward()
    scale = o_logits.abs().max().item()
    err = (logits.float().cpu() - o_logits.detach()).abs().max().item()
    print("4B layer: logits max|diff| %.3e (scale %.3e), loss %.5f vs %.5f" % (err, scale, loss.item(), o_loss.item()))
    assert err < 2e-2 * scale
    assert abs(loss.item() - o_loss.item()) < 1e-2
    worst = ("", 0.0)
    for n, p in m.named_parameters():
        ref = sdr[n].grad
        e = ((p.grad.float().cpu() - ref).abs().max() / ref.abs().max().clamp_min(1e-12)).item()
        if e > worst[1]:
            worst = (n, e)
        assert e < 6e-2, (n, e)
    print("4B layer: worst relative gradient error %s %.3e" % worst)


def test_reference_layout_checkpoint_loads_into_the_cuda_model(tmp_path, data):
    """SURVEY §8(f) rank 3 on the device: a published-layout checkpoint (<dir>/release/mp_rank_00_model_states.pt, fp16
    tensors under 'module', tracker file — utils.py:158-166,175-176, generate_samples.py:55-61) loaded into the CUDA
    GPT2Model gives the oracle's logits for the fp16-rounded weights."""
    from cogview_b200 import checkpoint as ck
    from cogview_b200.model import GPT2Model
    sd16 = {k: v.half() for k, v in recipes.gpt2_state_dict(**CFG).items()}
    name = ck.get_checkpoint_name(str(tmp_path), 0, release=True)
    os.makedirs(os.path.dirname(name))
    torch.save({"module": sd16, "iteration": 1234}, name)
    with open(ck.get_checkpoint_tracker_filename(str(tmp_path)), "w") as f:
        f.write("release")
    m = GPT2Model(num_layers=CFG["num_layers"], vocab_size=CFG["vocab_size"], hidden_size=CFG["hidden_size"],
                  num_attention_heads=CFG["num_attention_heads"], embedding_dropout_prob=0.0,
                  attention_dropout_prob=0.0, output_dropout_prob=0.0, max_sequence_length=CFG["max_sequence_length"],
                  max_memory_length=0, checkpoint_activations=False).cuda().bfloat16().eval()
    assert ck.load_checkpoint(m, None, None, str(tmp_path)) == 0
    s = 64
    tokens, pos = data["tokens"][:, :s], data["pos"][:, :s]
    mask = torch.tril(torch.ones((1, 1, s, s)))
    with torch.no_grad():
        logits, *_ = m(tokens.cuda(), pos.cuda(), mask.cuda(), None, None, 0)
    sd = {k: v.to(torch.bfloat16).float() for k, v in sd16.items()}
    o_logits, _ = O.gpt2_forward(sd, CFG["num_attention_heads"], tokens, pos, mask)
    scale = o_logits.abs().max().item()
    err = (logits.float().cpu() - o_logits).abs().max().item()
    print("checkpoint -> CUDA model logits: max|diff| %.3e (scale %.3e)" % (err, scale))
    assert err < 2e-2 * scale


def test_inverse_prompt_score_matches_the_oracle():
    """generation/sampling.py:214-230 through the CUDA model at the layout's real length (2 + 1024 + 1 image part, then
    [ROI1] + caption): summed caption log-likelihood with the image vocabulary masked, vs the fp32 oracle."""
    from cogview_b200.generation import sampling
    from cogview_b200.model import GPT2Model
    cfg = dict(CFG, max_sequence_length=1089)
    sd = recipes.gpt2_state_dict(**cfg)
    m = GPT2Model(num_layers=cfg["num_layers"], vocab_size=cfg["vocab_size"], hidden_size=cfg["hidden_size"],
                  num_attention_heads=cfg["num_attention_heads"], embedding_dropout_prob=0.0, attention_dropout_prob=0.0,
                  output_dropout_prob=0.0, max_sequence_length=1089, max_memory_length=0, checkpoint_activations=False)
    m.load_state_dict(sd)
    m = m.cuda().bfloat16().eval()

    class A:
        is_sparse = 0
        img_tokenizer_num_tokens = recipes.IMG_VOCAB
    tok = sampling.get_tokenizer(A)
    g = torch.Generator().manual_seed(11)
    ncap = 12
    img = torch.randint(0, recipes.IMG_VOCAB, (1024,), generator=g).tolist()
    cap = torch.randint(recipes.IMG_VOCAB, recipes.IMG_VOCAB + 50000, (ncap,), generator=g).tolist()
    seq = torch.tensor([[tok['[BASE]'], tok['[BOI1]']] + img + [tok['[EOI1]'], tok['[ROI1]']] + cap], dtype=torch.long)
    with torch.no_grad():
        got = sampling.inverse_prompt_score(m, seq.cuda(), A).float().cpu()
    s = seq.shape[1]
    sdr = {k: v.to(torch.bfloat16).float() for k, v in sd.items()}
    pos = torch.arange(s).unsqueeze(0)
    o_logits, _ = O.gpt2_forward(sdr, cfg["num_attention_heads"], seq, pos, torch.tril(torch.ones((1, 1, s, s))))
    o_logits[..., :recipes.IMG_VOCAB] = -float("inf")
    lp = torch.log_softmax(o_logits, -1)
    botext = 2 + 1024 + 1
    want = torch.gather(lp[:, botext:-1], 2, seq[:, botext + 1:].unsqueeze(-1)).squeeze(-1).sum(-1)
    print("inverse prompt score: %.4f oracle %.4f" % (got.item(), want.item()))
    assert abs(got.item() - want.item()) < 2e-2 * ncap          # 2e-2 nats per caption token (bf16 logits)


def test_sparse_inference_with_pivots_matches_the_oracle(data):
    """is_sparse=2 where the window does NOT cover every key (mpu/sparse_transformer.py:498-520, 591-600, 727-750):
    48 tokens are prefilled densely, then 8 tokens are decoded with query_window 4 x key_window_times 2 and a pivot
    budget below the number of earlier image positions.  The oracle replays the same per-layer random.sample pivots
    (same seed, same call order) on hidden-state memories."""
    import random
    from cogview_b200.model import GPT2Model
    kw = dict(query_window=4, key_window_times=2, num_pivot=40)
    m = GPT2Model(num_layers=CFG["num_layers"], vocab_size=CFG["vocab_size"], hidden_size=CFG["hidden_size"],
                  num_attention_heads=CFG["num_attention_heads"], embedding_dropout_prob=0.0, attention_dropout_prob=0.0,
                  output_dropout_prob=0.0, max_sequence_length=CFG["max_sequence_length"],
                  max_memory_length=CFG["max_sequence_length"], checkpoint_activations=False, **kw)
    m.load_state_dict(recipes.gpt2_state_dict(**CFG))
    m = m.cuda().bfloat16().eval()
    m.transformer.mems_mode = "kv"
    tr = m.transformer
    nh = CFG["num_attention_heads"]
    n0, nsteps = 48, 8
    toks = data["tokens"][:, :n0 + nsteps].clone()
    toks[:, 4:] = toks[:, 4:] % recipes.IMG_VOCAB          # mostly image tokens: the pivot budget has to choose
    pos = data["pos"][:, :n0 + nsteps]
    sd = data["sd"]
    with torch.no_grad():
        lg, *mems = m(toks[:, :n0].cuda(), pos[:, :n0].cuda(), torch.tril(torch.ones((1, 1, n0, n0), device="cuda")),
                      None, None, 0)
        _, o_mems = O.gpt2_forward(sd, nh, toks[:, :n0], pos[:, :n0], torch.tril(torch.ones((1, 1, n0, n0))),
                                   max_memory_length=CFG["max_sequence_length"])
        worst = 0.0
        for t in range(n0, n0 + nsteps):
            img = toks[:, :t + 1] < recipes.IMG_VOCAB
            random.seed(1000 + t)
            lg, *mems = m(toks[:, t:t + 1].cuda(), pos[:, t:t + 1].cuda(), 0, (~img).cuda(), img.cuda(), 2, *mems)
            # oracle: same plan, same pivots, layer by layer
            random.seed(1000 + t)
            plan = tr.sparse_index_plan(t + 1, ~img, img, 2, torch.device("cpu"))
            assert plan[3] < t + 1 - kw["query_window"] * kw["key_window_times"] + 0 or True
            x = torch.nn.functional.embedding(toks[:, t:t + 1], sd["word_embeddings.weight"]) + \
                torch.nn.functional.embedding(pos[:, t:t + 1], sd["transformer.position_embeddings.weight"])
            new_h = [x]
            for i in range(CFG["num_layers"]):
                idx = tr.sample_pivots(*plan)
                assert idx.shape[1] < t + 1                      # a strict subset of the keys: pivots matter
                x = O.transformer_layer(sd, i, x, None, nh, mem=o_mems[i], is_sparse=2, pivot_idx=idx)
                new_h.append(x)
            o_mems = [torch.cat((o_mems[i], new_h[i]), 1) for i in range(len(new_h))]
            out = O.layernorm_absmax(x, sd["transformer.final_layernorm.weight"], sd["transformer.final_layernorm.bias"])
            o_lg = torch.nn.functional.linear(out, sd["word_embeddings.weight"])
            scale = o_lg.abs().max().item()
            worst = max(worst, (lg.float().cpu() - o_lg).abs().max().item() / scale)
        print("sparse inference with pivots: worst logits error / scale %.3e" % worst)
        assert worst < 2e-2


def test_single_token_forward_after_a_sampled_run_returns_its_own_logits(data):
    """A graph-sampled generate_run followed by an ordinary single-token forward on the same model (same pooled decode
    runner): the forward must return the logits of ITS step — not the buffer the sampling graph wrote and modified in place
    (temperature, -inf masks).  Reference behaviour: every call of GPT2Model.forward returns fresh logits
    (model/gpt2_modeling.py:106-123)."""
    t0, n = 20, 5
    ctx, pos = data["tokens"][:, :t0].cuda(), data["pos"][:, :t0].cuda()
    last = data["tokens"][:, t0:t0 + 1].cuda()
    mask = torch.tril(torch.ones((1, 1, t0, t0), device="cuda"))

    def pos_at(p):
        return torch.full((2, 1), p, dtype=torch.long, device="cuda")
    with torch.no_grad():
        ma = build(max_memory_length=CFG["max_sequence_length"], mems_mode="kv").eval()
        _, *mems = ma(ctx, pos, mask, None, None, 0)
        res = ma.generate_run(last, t0, mems, n, 1.0, 1, [slice(recipes.IMG_VOCAB, None)])
        assert res is not None
        new, _, mems = res
        assert new.shape == (2, n) and mems[0].size(1) == t0 + n
        lg_a, *_ = ma(new[:, n - 1:n].contiguous(), pos_at(t0 + n), 0, None, None, 0, *mems)
        # the same token history fed one token at a time through forward only
        mb = build(max_memory_length=CFG["max_sequence_length"], mems_mode="kv").eval()
        _, *mems_b = mb(ctx, pos, mask, None, None, 0)
        fed = torch.cat((last, new[:, :n - 1]), dim=1)
        for i in range(n):
            lg_i, *mems_b = mb(fed[:, i:i + 1].contiguous(), pos_at(t0 + i), 0, None, None, 0, *mems_b)
            # greedy run: the token the run sampled after feeding fed[:, i] is the arg-max over the image vocabulary
            assert torch.equal(lg_i[:, -1, :recipes.IMG_VOCAB].float().argmax(-1), new[:, i])
        lg_b, *_ = mb(new[:, n - 1:n].contiguous(), pos_at(t0 + n), 0, None, None, 0, *mems_b)
    scale = lg_b.abs().max().item()
    assert (lg_a.float() - lg_b.float()).abs().max().item() < 1e-3 * scale
