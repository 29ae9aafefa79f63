"""CPU: the restatement of sparse training attention with attention-probability dropout
(oracle/sparse_dropout_oracle.py; mpu/sparse_transformer.py:675-725 with the dropout of :719-721) against
tests/golden/sparse_dropout.npz, the UNMODIFIED reference's output under a seeded keep tensor
(oracle/make_sparse_dropout_golden.py).  The keep tensor is re-derived from its stored seed.  With an all-ones keep
tensor and p = 0 the restatement must be bitwise the dropout-free oracle, for the attention and for a whole layer."""
import os

import numpy as np
import torch

from oracle import cogview_oracle as O
from oracle import recipes
from oracle import sparse_dropout_oracle as SD


def _inputs(golden_dir):
    g = np.load(os.path.join(golden_dir, "sparse_dropout.npz"), allow_pickle=False)
    b, nh, s, hn, w, times, n_piv = [int(x) for x in g["dims"]]
    gen = torch.Generator().manual_seed(int(g["seed"]))
    q, k, v = (torch.randn((b, nh, s, hn), generator=gen) for _ in range(3))
    pivot_idx = torch.from_numpy(g["pivot_idx"])
    gcount = s // w
    tmp = torch.tril(1 - torch.block_diag(*torch.ones((gcount - times + 1, w, w))))
    rmask = torch.nn.functional.pad(tmp, (0, (times - 1) * w, (times - 1) * w, 0))
    pam = rmask.expand(b, s, s).gather(dim=-1, index=pivot_idx.unsqueeze(1).expand(b, s, n_piv))
    p = float(g["p"])
    kg = torch.Generator().manual_seed(int(g["keep_seed"]))
    keep = (torch.rand((b, nh, s, n_piv + w * times), generator=kg) >= p).float()
    return g, (q, k, v, pivot_idx, pam, w, times), keep, p


def test_oracle_sparse_dropout_matches_reference_golden(golden_dir):
    g, args, keep, p = _inputs(golden_dir)
    out = SD.sparse_attention(*args, keep, p)
    assert np.allclose(out.numpy()[:, :, ::7], g["sparse_train_dropout"], atol=1e-5)
    # the keep tensor matters: without it the output is far from the fixture
    plain = O.sparse_attention(*args)
    assert not np.allclose(plain.numpy()[:, :, ::7], g["sparse_train_dropout"], atol=1e-2)


def test_oracle_all_ones_keep_at_p0_is_bitwise_unchanged(golden_dir):
    _, args, keep, _ = _inputs(golden_dir)
    plain = O.sparse_attention(*args)
    ones = SD.sparse_attention(*args, torch.ones_like(keep), 0.0)
    assert torch.equal(plain, ones)


def test_layer_with_all_ones_keep_at_p0_is_bitwise_the_oracle_layer():
    b, s, w, times, n_piv, heads = 2, 256, 64, 2, 48, 4
    sd = recipes.gpt2_state_dict(seed=21, num_layers=1, vocab_size=512, hidden_size=256, num_attention_heads=heads,
                                 max_sequence_length=s)
    g = torch.Generator().manual_seed(3)
    x = torch.randn((b, s, 256), generator=g)
    pivot_idx = torch.stack([torch.randperm(s, generator=g)[:n_piv] for _ in range(b)])
    gcount = s // w
    tmp = torch.tril(1 - torch.block_diag(*torch.ones((gcount - times + 1, w, w))))
    rmask = torch.nn.functional.pad(tmp, (0, (times - 1) * w, (times - 1) * w, 0))
    pam = rmask.expand(b, s, s).gather(dim=-1, index=pivot_idx.unsqueeze(1).expand(b, s, n_piv))
    ref = O.transformer_layer(sd, 0, x, pam, heads, is_sparse=1, pivot_idx=pivot_idx, query_window=w,
                              key_window_times=times)
    ones = torch.ones((b, heads, s, n_piv + w * times))
    got = SD.transformer_layer(sd, 0, x, pam, heads, pivot_idx, w, times, ones, 0.0)
    assert torch.equal(ref, got)
