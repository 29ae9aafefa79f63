"""TEST INFRASTRUCTURE — golden fixture of sparse training attention with attention-probability dropout.
Runs ONLY where the reference can be placed under oracle/_ref (oracle/build_ref.py).

  python oracle/make_sparse_dropout_golden.py

Runs the UNMODIFIED reference's sparse_attention (mpu/sparse_transformer.py:675-725) at the shape of the attention
fixture of oracle/make_golden.py (s = 512, w = 64, times = 3, 96 pivots, 2 x 3 heads) with, as `attention_dropout`,
a callable that multiplies by a seeded keep tensor and scales by 1/(1-p) (the harness's no-op fork() stands in for the
RNG tracker, :719-721).  Asserts oracle/sparse_dropout_oracle.py reproduces it (fp32) and writes
tests/golden/sparse_dropout.npz: the output (every 7th head dimension, as attention.npz) and the seeds — the inputs
and the keep tensor are re-derived from them.
"""
import os
import random
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import build_ref, ref_harness  # noqa: E402
from oracle import sparse_dropout_oracle as SD  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
SEED, KEEP_SEED, P = 7, 2024, 0.1
DIMS = (2, 3, 512, 64, 64, 3, 96)        # b, nh, s, hn, w, times, n_piv
TXT_N = (48, 20)


def inputs(seed=SEED, keep_seed=KEEP_SEED, p=P, dims=DIMS):
    """q, k, v, pivot_idx, the reference's gathered pivot mask and the keep tensor, all from the seeds."""
    b, nh, s, hn, w, times, n_piv = dims
    g = torch.Generator().manual_seed(seed)
    q, k, v = (torch.randn((b, nh, s, hn), generator=g) for _ in range(3))
    random.seed(1234)
    pivot_idx = torch.stack([
        torch.cat((torch.arange(0, TXT_N[i]),
                   torch.tensor(random.sample(range(TXT_N[i], s), n_piv - TXT_N[i]), dtype=torch.long)))
        for i in range(b)])
    gcount = s // w
    tmp = torch.tril(1 - torch.block_diag(*torch.ones((gcount - times + 1, w, w))))
    rmask = torch.nn.functional.pad(tmp, (0, (times - 1) * w, (times - 1) * w, 0))
    pam = rmask.expand(b, s, s).gather(dim=-1, index=pivot_idx.unsqueeze(1).expand(b, s, n_piv))
    kg = torch.Generator().manual_seed(keep_seed)
    keep = (torch.rand((b, nh, s, n_piv + w * times), generator=kg) >= p).float()
    return q, k, v, pivot_idx, pam, keep


def main():
    os.makedirs(GOLD, exist_ok=True)
    torch.set_num_threads(8)
    if not build_ref.build():
        raise SystemExit("make_sparse_dropout_golden: the reference is not available under oracle/_ref")
    st = ref_harness.load()["sparse_transformer"]
    b, nh, s, hn, w, times, n_piv = DIMS
    q, k, v, pivot_idx, pam, keep = inputs()
    r = st.sparse_attention(q, k, v, pivot_idx, pam, w, times, lambda probs: probs * keep / (1.0 - P))
    o = SD.sparse_attention(q, k, v, pivot_idx, pam, w, times, keep, P)
    err = (o - r).abs().max().item()
    print("sparse_attention with dropout %.1f: restatement vs reference max|diff| %.3e (scale %.3e)" % (
        P, err, r.abs().max().item()))
    assert err <= 1e-5 * max(1.0, r.abs().max().item())
    r0 = st.sparse_attention(q, k, v, pivot_idx, pam, w, times, None)
    print("  dropout changes the output by %.3e" % (r - r0).abs().max().item())
    np.savez_compressed(os.path.join(GOLD, "sparse_dropout.npz"), seed=np.int64(SEED), keep_seed=np.int64(KEEP_SEED),
                        p=np.float64(P), dims=np.array(DIMS), pivot_idx=pivot_idx.numpy(),
                        sparse_train_dropout=r.numpy()[:, :, ::7])
    print("written", os.path.join(GOLD, "sparse_dropout.npz"))


if __name__ == "__main__":
    main()
