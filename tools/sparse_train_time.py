"""Cost of attention-probability dropout in sparse training attention (is_sparse = 1).

  python tools/sparse_train_time.py [--layers 4] [--steps 5]

1. cv_attn_sparse_fwd / _bwd at the CogView-sr shape (b = 2, 40 heads, s = 4096, w = 128, times = 6, 768 pivots) at
   p = 0 and p = 0.1, alternated, CUDA-event timed (median, L2 flushed before every call); the sparse keep-bit kernel
   on its own from torch.profiler's device times.
2. A training step (forward + loss + backward) of a GPT2Model at the 4B width (h = 2560, 40 heads) with is_sparse = 1,
   checkpoint_activations, attention_dropout_prob 0 and 0.1 (other dropouts 0), alternated.
Prints the card name and power limit first: both are part of the numbers."""
import argparse
import os
import random
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from cogview_b200 import ops  # noqa: E402


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip()
    except OSError:
        return torch.cuda.get_device_name(0) + ", power limit unknown"


def median_us(fns, n, flush):
    """Times every fn of `fns` n times, interleaved; returns the median of each in microseconds."""
    ts = [[] for _ in fns]
    for _ in range(n):
        for i, fn in enumerate(fns):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts[i].append(a.elapsed_time(b) * 1e3)
    return [sorted(t)[len(t) // 2] for t in ts]


def attention_calls(n):
    b, heads, s, w, times, n_piv = 2, 40, 4096, 128, 6, 768
    h = heads * 64
    g = torch.Generator(device="cuda").manual_seed(0)
    qkv = torch.randn((b, s, 3 * h), generator=g, device="cuda").bfloat16()
    d_out = torch.randn((b, s, h), generator=g, device="cuda").bfloat16()
    q, k, v = qkv[..., :h], qkv[..., h:2 * h], qkv[..., 2 * h:]
    random.seed(1)
    piv = torch.stack([torch.cat((torch.arange(64), torch.tensor(random.sample(range(64, s), n_piv - 64))))
                       for _ in range(b)]).cuda()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    drop = (0.1, 1234, 3)
    out0, lse0 = ops.attn_sparse_fwd(q, k, v, heads, piv, w, times, want_lse=True)
    out1, lse1, mask = ops.attn_sparse_fwd(q, k, v, heads, piv, w, times, want_lse=True, dropout=drop)
    fwd = [lambda: ops.attn_sparse_fwd(q, k, v, heads, piv, w, times, want_lse=True),
           lambda: ops.attn_sparse_fwd(q, k, v, heads, piv, w, times, want_lse=True, dropout=drop)]
    bwd = [lambda: ops.attn_sparse_bwd(q, k, v, out0, d_out, lse0, heads, piv, w, times),
           lambda: ops.attn_sparse_bwd(q, k, v, out1, d_out, lse1, heads, piv, w, times, dropout_p=0.1,
                                       drop_mask=mask)]
    median_us(fwd + bwd, 3, flush)                   # warm-up
    f0, f1, b0, b1 = median_us(fwd + bwd, n, flush)
    # the keep-bit kernel alone: device time from the profiler (the forward with dropout launches it)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(10):
            fwd[1]()
        torch.cuda.synchronize()
    mk = [e for e in prof.key_averages() if "attn_dropout_mask_kernel" in e.key]
    mask_us = (sum(e.device_time_total for e in mk) / sum(e.count for e in mk)) if mk else float("nan")
    print("sparse attention b=%d heads=%d s=%d w=%d x%d pivots=%d (median of %d, alternated):" % (
        b, heads, s, w, times, n_piv, n))
    print("  forward  p=0 %8.1f us   p=0.1 %8.1f us   (+%.1f %%)" % (f0, f1, 100 * (f1 / f0 - 1)))
    print("  backward p=0 %8.1f us   p=0.1 %8.1f us   (+%.1f %%)" % (b0, b1, 100 * (b1 / b0 - 1)))
    print("  keep-bit kernel alone %.1f us per call; keep bits %.1f MB" % (mask_us, mask.numel() * 4 / 2 ** 20))


def training_steps(layers, n):
    from cogview_b200 import mpu
    from cogview_b200.model import GPT2Model
    from oracle import recipes
    b, s, h, heads = 1, 4096, 2560, 40
    models = {}
    for p in (0.0, 0.1):
        torch.manual_seed(0)
        models[p] = GPT2Model(num_layers=layers, vocab_size=58240, hidden_size=h, num_attention_heads=heads,
                              embedding_dropout_prob=0.0, attention_dropout_prob=p, output_dropout_prob=0.0,
                              max_sequence_length=s, max_memory_length=0, checkpoint_activations=True,
                              checkpoint_num_layers=1, query_window=128, key_window_times=6,
                              num_pivot=768).cuda().bfloat16().train()
    tokens = recipes.text_image_tokens(b, 64, s - 64, seed=0)
    labels = torch.roll(tokens, -1, dims=1).cuda()
    img = tokens < recipes.IMG_VOCAB
    args = (tokens.cuda(), torch.arange(s).unsqueeze(0).expand(b, -1).contiguous().cuda(),
            torch.tril(torch.ones((1, 1, s, s), device="cuda")), (~img).cuda(), img.cuda(), 1)

    def step(m):
        def run():
            m.zero_grad(set_to_none=True)
            logits, *_ = m(*args)
            mpu.vocab_parallel_cross_entropy(logits.contiguous().float(), labels).mean().backward()
        return run
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    fns = [step(models[0.0]), step(models[0.1])]
    median_us(fns, 2, flush)
    t0, t1 = median_us(fns, n, flush)
    print("training step, %d layers h=%d heads=%d s=%d b=%d, is_sparse=1, checkpointing (median of %d, alternated):" % (
        layers, h, heads, s, b, n))
    print("  attention_dropout_prob 0   %8.2f ms" % (t0 / 1e3))
    print("  attention_dropout_prob 0.1 %8.2f ms   (+%.2f ms, +%.1f %%; %.1f us per layer)" % (
        t1 / 1e3, (t1 - t0) / 1e3, 100 * (t1 / t0 - 1), (t1 - t0) / layers))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--layers", type=int, default=4)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--calls", type=int, default=20)
    a = ap.parse_args()
    print("card:", card())
    attention_calls(a.calls)
    training_steps(a.layers, a.steps)


if __name__ == "__main__":
    main()
