"""Host-side logic that needs no GPU: attention-mask recognition, sampling helpers, the sparse-inference index plan,
the weight-decay parameter split and the oracle's building blocks against plain PyTorch restatements of the
reference formulas (mpu/sparse_transformer.py:33-44, :172-176, :477-489, :498-520; generation/sampling.py:24-49,
:188-211; model/gpt2_modeling.py:122-146)."""
import random

import pytest
import torch

from oracle import cogview_oracle as O


def test_mask_to_sep_recognises_the_reference_mask_families():
    from cogview_b200.mpu.sparse_transformer import mask_to_sep
    s = 96
    tril = torch.tril(torch.ones((1, 1, s, s)))
    assert mask_to_sep(tril, s, s) == 0
    assert mask_to_sep(17, s, s) == 17 and mask_to_sep(torch.tensor([23]), s, s) == 23
    for sep in (5, 40, s):
        assert mask_to_sep(O.build_sep_mask(s, s, sep), s, s) == sep
    # memory columns (sk > sq): every memory position is visible, the rest is causal
    sq, sk = 8, 40
    assert mask_to_sep(O.build_sep_mask(sq, sk, 0), sq, sk) == 0
    assert mask_to_sep(O.build_sep_mask(sq, sk, 3), sq, sk) == 3
    bad = tril.clone()
    bad[0, 0, 10, 50] = 1.0                                   # not causal: no kernel for it -> loud failure
    with pytest.raises(NotImplementedError):
        mask_to_sep(bad, s, s)
    with pytest.raises(ValueError):
        mask_to_sep(torch.ones((2, 1, s, s)), s, s)


def test_build_sep_mask_matches_reference_construction():
    # mpu/sparse_transformer.py:477-489: m = tril(ones); m[:, :sep] = 1; memory columns prepended as ones
    for sq, sk, sep in ((16, 16, 0), (16, 16, 7), (6, 20, 0), (6, 20, 4)):
        m = torch.ones((1, sq, sk)).tril(diagonal=sk - sq)
        m[0, :, :sep + (sk - sq)] = 1
        assert torch.equal(O.build_sep_mask(sq, sk, sep), m.unsqueeze(1))


def test_top_k_top_p_filtering():
    from cogview_b200.generation import sampling
    g = torch.Generator().manual_seed(0)
    logits = torch.randn((1, 500), generator=g)
    out = sampling.top_k_logits(logits.clone(), top_k=20)
    kept = torch.isfinite(out[0])
    assert kept.sum().item() == 20 and torch.equal(out[0][kept], logits[0][kept])
    assert logits[0][kept].min() >= logits[0][~kept].max()
    assert torch.equal(out, O.top_k_logits(logits.clone(), top_k=20))
    # nucleus: the kept set is the smallest prefix of the sorted distribution whose mass exceeds top_p
    out = sampling.top_k_logits(logits.clone(), top_k=0, top_p=0.7)
    kept = torch.isfinite(out[0])
    p = torch.softmax(logits[0], -1)
    mass = p[kept].sum().item()
    assert mass > 0.7 and mass - p[kept].min().item() <= 0.7 + 1e-6
    assert p[kept].min() >= p[~kept].max()


def test_shrink_beams_and_interlacing_marks():
    from cogview_b200.generation import sampling
    tokens = torch.arange(12).view(3, 4)
    mems = [torch.arange(3 * 2 * 5, dtype=torch.float32).view(3, 2, 5) for _ in range(2)]
    t, m, sc = sampling.shrink_beams(tokens, mems, 3, [0.1, 0.9, 0.3])
    assert t is tokens and sc == [0.1, 0.9, 0.3]                      # beam count unchanged: nothing happens
    t, m, sc = sampling.shrink_beams(tokens, mems, 1, torch.tensor([0.1, 0.9, 0.3]))
    assert torch.equal(t, tokens[1:2]) and all(torch.equal(a, b[1:2]) for a, b in zip(m, mems)) and sc == [0]
    seq = [5, -1, -1, 7, -1, -1, -1, -1]
    sampling.add_interlacing_beam_marks(seq, nb=3, period=2)
    # after `period` consecutive generated slots nb alternates 3 -> 4 -> 3 (nb += (nb % 2) * 2 - 1); a context
    # token resets the run counter
    assert seq == [5, -3, -3, 7, -4, -4, -3, -3]


def test_masks_and_position_ids():
    from cogview_b200.generation import sampling
    data = torch.zeros((3, 10), dtype=torch.long)
    am, lm, pos = sampling.get_masks_and_position_ids(data)
    assert am.shape == (1, 1, 10, 10) and torch.equal(am[0, 0], torch.tril(torch.ones(10, 10)))
    assert torch.equal(lm, torch.ones(3, 10)) and torch.equal(pos, torch.arange(10).expand(3, 10))


def test_sparse_inference_index_plan_and_pivot_sampling():
    from cogview_b200.mpu.sparse_transformer import GPT2ParallelTransformer
    w, times, num_pivot, max_seq = 8, 3, 40, 100
    plan_of = GPT2ParallelTransformer.sparse_index_plan
    sample = GPT2ParallelTransformer.sample_pivots

    class Cfg:
        query_window, key_window_times, max_sequence_length = w, times, max_seq
    Cfg.num_pivot = num_pivot
    b, key_length = 2, 70
    txt = torch.zeros((b, key_length), dtype=torch.bool)
    txt[0, :6] = True
    txt[1, :9] = True
    img = ~txt
    window_idx, img_idx, txt_idx, n_piv = plan_of(Cfg, key_length, txt, img, b, torch.device("cpu"))
    left = key_length - times * w
    assert torch.equal(window_idx, torch.arange(left, key_length).expand(b, -1))
    assert [len(t) for t in txt_idx] == [6, 9] and [len(t) for t in img_idx] == [left - 6, left - 9]
    assert n_piv == 9 + int((left - 9) * num_pivot / max_seq)
    random.seed(5)
    pw = sample(Cfg, window_idx, img_idx, txt_idx, n_piv)
    assert pw.shape == (b, n_piv + times * w)
    random.seed(5)                                           # the reference's RNG: Python random.sample, per sample
    for i in range(b):
        picks = random.sample(range(len(img_idx[i])), k=n_piv - len(txt_idx[i]))
        want = torch.cat((txt_idx[i], img_idx[i][torch.tensor(picks, dtype=torch.long)], window_idx[i]))
        assert torch.equal(pw[i], want)
        assert len(set(pw[i].tolist())) == pw.shape[1]       # pivots, window: disjoint positions


def test_oracle_building_blocks_against_plain_formulas():
    g = torch.Generator().manual_seed(1)
    x = torch.randn((5, 64), generator=g) * 50
    w, bias = torch.randn(64, generator=g), torch.randn(64, generator=g)
    # LayerNorm.forward (mpu/sparse_transformer.py:40-44): F.layer_norm(x / (max|x| / 8))
    ref = torch.nn.functional.layer_norm(x / (x.abs().max().detach() / 8), (64,), w, bias, 1e-5)
    assert torch.allclose(O.layernorm_absmax(x, w, bias), ref, atol=1e-6)
    # gelu_impl (:172-176)
    y = torch.randn(100, generator=g) * 3
    ref = 0.5 * y * (1.0 + torch.tanh(0.7978845608028654 * y * (1.0 + 0.044715 * y * y)))
    assert torch.allclose(O.gelu(y), ref, atol=1e-6)
    # vocab_parallel_cross_entropy at MP = 1 (mpu/cross_entropy.py:26-77) == F.cross_entropy
    logits, tgt = torch.randn((4, 7, 33), generator=g), torch.randint(0, 33, (4, 7), generator=g)
    ref = torch.nn.functional.cross_entropy(logits.view(-1, 33), tgt.view(-1), reduction="none").view(4, 7)
    assert torch.allclose(O.vocab_parallel_cross_entropy(logits, tgt), ref, atol=1e-5)
    # standard_attention (:652-673): (q / sqrt(hn)) k^T * mask - 10000 (1 - mask), softmax, @ v
    q, k, v = (torch.randn((2, 3, 16, 8), generator=g) for _ in range(3))
    m = O.build_sep_mask(16, 16, 4)
    s = torch.matmul(q / 8 ** 0.5, k.transpose(-1, -2)) * m - 10000.0 * (1 - m)
    assert torch.allclose(O.standard_attention(q, k, v, m), torch.matmul(torch.softmax(s, -1), v), atol=1e-5)


def test_weight_decay_parameter_groups():
    """gpt2_get_params_for_weight_decay_optimization (model/gpt2_modeling.py:122-146): LayerNorm parameters and all
    biases go to the no-decay group, everything else decays; every parameter appears exactly once."""
    from cogview_b200.model import GPT2Model, gpt2_get_params_for_weight_decay_optimization
    m = GPT2Model(num_layers=2, vocab_size=128, hidden_size=64, num_attention_heads=1, embedding_dropout_prob=0.,
                  attention_dropout_prob=0., output_dropout_prob=0., max_sequence_length=32, max_memory_length=0,
                  checkpoint_activations=False)
    decay, no_decay = gpt2_get_params_for_weight_decay_optimization(m)
    assert 'weight_decay' not in decay and no_decay['weight_decay'] == 0.0
    ids = [id(p) for p in decay['params'] + no_decay['params']]
    assert len(ids) == len(set(ids)) == len(list(m.parameters()))
    names = {id(p): n for n, p in m.named_parameters()}
    for p in no_decay['params']:
        assert names[id(p)].endswith('bias') or 'layernorm' in names[id(p)].lower(), names[id(p)]
    for p in decay['params']:
        assert names[id(p)].endswith('weight') and 'layernorm' not in names[id(p)].lower(), names[id(p)]


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the reference's own modules from oracle/_ref on the host cores; the oracle port
    when build() could not place them there) on the tiny configuration: one JSON line with the contract's keys,
    `impl = reference`, a `cpu_baseline` describing the run and a zero-copy `e2e`."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--model", "tiny",
                        "--steps", "1", "--warmup", "0", "--gen-tokens", "16"], capture_output=True, text=True,
                       timeout=300, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "tokens/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["kind"] in ("reference", "port")
    ref_here = os.path.isdir(os.path.join(root, "oracle", "_ref", "mpu"))
    assert d["cpu_baseline"]["kind"] == ("reference" if ref_here else "port")
    assert d["cpu_baseline"]["cores"] >= 1 and "workload" in d["config"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_bench_reference_arm_under_torchrun_does_not_wait_for_a_rendezvous():
    """The driver launches `bench.py --impl reference --gpus N` under torchrun for N > 1: rank 0 alone does the work and
    prints the line, the other ranks exit 0.  The reference's mpu needs a process group — it must be a private one (a
    file store): with TORCHELASTIC_USE_AGENT_STORE in the environment an env:// or tcp:// group would try to join the
    agent's store as a client and block until its timeout."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29571", os.path.join(root, "bench.py"), "--impl",
                        "reference", "--gpus", "2", "--model", "tiny", "--steps", "1", "--warmup", "0", "--gen-tokens", "16"],
                       capture_output=True, text=True, timeout=240, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and d["value"] > 0


def test_filling_sequence_sparse_run_keeps_index_masks_current():
    """filling_sequence with is_sparse == 2: a stretch of generate slots goes through model.generate_run(sparse=...) with the
    full token history; the text / image index masks handed to the next host-loop call must cover the tokens the run
    appended (mpu/sparse_transformer.py:498-520 indexes them by position)."""
    from cogview_b200.generation import sampling

    class A:
        temperature, top_k, top_p, is_sparse = 1.0, 0, 0.0, 2
        img_tokenizer_num_tokens = 8192
    tok = sampling.get_tokenizer(A)
    V = tok.num_tokens
    calls = {"run": [], "fwd": []}

    class StandIn:
        def __call__(self, tokens, position_ids, attention_mask, txt, img, is_sparse, *mems):
            assert is_sparse == 2 and txt is not None and img is not None
            t_prev = mems[0].shape[1] if mems else 0
            assert txt.shape == img.shape and txt.shape[1] == t_prev + tokens.shape[1]      # masks cover every position
            calls["fwd"].append(tokens.shape)
            b, sq = tokens.shape
            g = torch.Generator().manual_seed(t_prev)
            logits = torch.randn((b, sq, V), generator=g)
            mem = torch.zeros((b, t_prev + sq, 1))
            return (logits, mem)

        def generate_run(self, last_tokens, first_pos, mems, n_steps, temperature, top_k, invalid_slices, sparse=None):
            assert sparse is not None and sparse["n_img"] == 8192
            assert sparse["tokens"].shape[1] == mems[0].shape[1] + 1                        # history incl. the fed token
            calls["run"].append(n_steps)
            b = last_tokens.shape[0]
            new = torch.arange(n_steps).unsqueeze(0).expand(b, -1) % 8192
            mem = torch.zeros((b, mems[0].shape[1] + n_steps, 1))
            return new, torch.zeros(b), [mem]

    text = list(range(8192, 8192 + 6))
    seq = [tok['[ROI1]']] + text + [tok['[BASE]'], tok['[BOI1]']] + [-2] * 7 + [tok['[EOI1]']] + [-1]
    out = sampling.filling_sequence(StandIn(), torch.tensor(seq, dtype=torch.long), A)
    assert out.shape[1] == len(seq)
    assert calls["run"] == [6]                 # the first of the seven -2 slots expands the beams on the host
    # the context call, then (after the device run and the provided [EOI1]) one host-loop call fed with the two newest
    # tokens — its masks were checked above against the memory length that includes the run's six tokens
    assert len(calls["fwd"]) == 2 and calls["fwd"][-1][1] == 2
