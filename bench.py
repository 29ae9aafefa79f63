#!/usr/bin/env python
"""bench.py — CogView-base 4B hot path on B200 (BASELINE.json metric: tokens/sec, train + AR sample).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload sample|train|both]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Headline line (`value`, `e2e`): BASELINE.json configs[1] — 4B (48 L, d=2560, 40 heads, V=58240), 1089-token
sequences, bf16, autoregressive sampling through the reference-facing API (generation.sampling.filling_sequence
over GPT2Model): one step = prefill a 65-token context and generate 1024 image tokens for a batch of 4 beams
(scripts/text2image.sh defaults).  The same JSON line carries a `train` object for configs[2] (one optimizer
step on 4 x 1088 tokens per GPU: forward, vocab cross-entropy, backward, DP gradient all-reduce, fused AdamW).
Synthetic tokens, random-init weights (no network for checkpoints).  `--impl reference` times the reference's
own modules (oracle/_ref, placed by oracle/build_ref.py; hidden-state `mems` semantics) on the host cores — or the
oracle port when oracle/_ref is absent.  The driver's record keeps only the contract keys of the JSON line, so the
training / VQ-VAE results are also summarised inside `config` (`config.train`, `config.vqvae`).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

MODEL_4B = dict(num_layers=48, vocab_size=58240, hidden_size=2560, num_attention_heads=40, max_sequence_length=1089)
MODEL_TINY = dict(num_layers=2, vocab_size=58240, hidden_size=256, num_attention_heads=4, max_sequence_length=1089)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="all", choices=["sample", "train", "vqvae", "both", "all"])
    ap.add_argument("--vq-batch", type=int, default=256)
    ap.add_argument("--batch", type=int, default=4, help="beams per GPU (sampling) / sequences per GPU (training)")
    ap.add_argument("--gen-tokens", type=int, default=1024)
    ap.add_argument("--model", default="4b", choices=["4b", "tiny"])
    ap.add_argument("--train-steps", type=int, default=None)
    ap.add_argument("--skip-cpu-baseline", action="store_true",
                    help="development only: leave out the host-core baseline leg (the default run includes it)")
    ap.add_argument("--dropout", type=float, default=0.1,
                    help="embedding/attention/hidden dropout of the training workload (reference scripts: 0.1)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step of each workload returned as DIR/<name>.npy "
                         "(float32; large outputs as a fixed seeded sample), to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours (the reference arm only samples timings)")
    return args


def measured_traffic(kernel):
    """DRAM bytes per launch from the committed ncu captures (profiles/r02_traffic.json, r01_traffic.json), or None."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        try:
            return json.load(open(os.path.join(ROOT, "profiles", name)))[kernel]["traffic_bytes_per_launch"]
        except Exception:
            continue
    return None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback (B200_PROFILING.md)")


# ----------------------------------------------------------------------------------------------------
# clocks during the timed region
# ----------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.thread = [], None, None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower() == "active"})
        busy = [x for x in sm if x > 0.5 * max(sm)] if sm else []
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------
# model / workload construction
# ----------------------------------------------------------------------------------------------------
def build_model(cfg, max_memory_length, device, dropout=0.0):
    from cogview_b200.model import GPT2Model
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.bfloat16)
    try:
        with torch.device(device):
            model = GPT2Model(num_layers=cfg["num_layers"], vocab_size=cfg["vocab_size"],
                              hidden_size=cfg["hidden_size"], num_attention_heads=cfg["num_attention_heads"],
                              embedding_dropout_prob=dropout, attention_dropout_prob=dropout,
                              output_dropout_prob=dropout, max_sequence_length=cfg["max_sequence_length"],
                              max_memory_length=max_memory_length, checkpoint_activations=False)
    finally:
        torch.set_default_dtype(old)
    return model


class SampleArgs:
    temperature = 1.0
    top_k = 200
    top_p = 0.0
    is_sparse = 0
    img_tokenizer_num_tokens = 8192


def make_template(nb, gen_tokens, seed):
    """'[ROI1] text [BASE] [BOI1] [MASK]*N' (generate_samples.py:204) as token ids; -nb marks generated slots."""
    from cogview_b200.generation import sampling
    tok = sampling.get_tokenizer(SampleArgs)
    g = torch.Generator().manual_seed(seed)
    text = torch.randint(8192, 58192, (62,), generator=g).tolist()
    seq = [tok['[ROI1]']] + text + [tok['[BASE]'], tok['[BOI1]']] + [-1] * gen_tokens
    sampling.add_interlacing_beam_marks(seq, nb=nb)
    return torch.tensor(seq, dtype=torch.long)


def param_count(model):
    return sum(p.numel() for p in model.parameters())


# ----------------------------------------------------------------------------------------------------
# timing helpers
# ----------------------------------------------------------------------------------------------------
def dist_ready():
    return torch.distributed.is_available() and torch.distributed.is_initialized()


def barrier():
    if dist_ready():
        torch.distributed.barrier()


def timed(fn, steps, warmup, device_index):
    """W untimed + K timed steps: barrier + sync on both sides, CUDA events on the launching stream, MAX over ranks."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    barrier()
    sampler = ClockSampler(device_index)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    barrier()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop()
    if dist_ready():
        t = torch.tensor([ms], device="cuda")
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms = t.item()
    return ms, clocks


def launches():
    from cogview_b200 import _lib
    return int(_lib.lib().cv_launch_count())


# ----------------------------------------------------------------------------------------------------
# sampling workload (configs[1])
# ----------------------------------------------------------------------------------------------------
def run_sample(args, cfg, world, rank, dev_index):
    from cogview_b200.generation import sampling
    torch.manual_seed(rank)            # weights and the sampling draws: the same run for the same arguments
    model = build_model(cfg, cfg["max_sequence_length"], "cuda").eval()
    nb = args.batch
    tmpl_host = make_template(nb, args.gen_tokens, seed=rank).pin_memory()
    tmpl_dev = tmpl_host.cuda()
    out_host = torch.empty((nb, tmpl_host.numel()), dtype=torch.long).pin_memory()
    holder = {}

    def step_dev():
        with torch.no_grad():
            holder["out"] = sampling.filling_sequence(model, tmpl_dev, SampleArgs)

    def step_e2e():
        with torch.no_grad():
            seq = tmpl_host.cuda(non_blocking=True)
            out = sampling.filling_sequence(model, seq, SampleArgs)
            out_host.copy_(out, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    tokens_per_step = nb * args.gen_tokens * world
    l0 = launches()
    ms_dev, clocks = timed(step_dev, args.steps, args.warmup, dev_index)
    outputs = dict(sample_tokens=holder["out"]) if args.dump_outputs else {}
    graph_nodes = 0
    kv = model.transformer._kv
    if kv is not None and getattr(kv, "runner", None) is not None:
        graph_nodes = kv.runner.graph_launches * kv.runner.replays
    n_launch = launches() - l0 + graph_nodes
    ms_e2e, _ = timed(step_e2e, args.steps, 1, dev_index)
    assert holder["out"].shape == (nb, tmpl_host.numel()) and int(holder["out"].min()) >= 0
    assert int(holder["out"][:, -args.gen_tokens:].max()) < 8192, "generated tokens must be image codes"
    res = dict(value=tokens_per_step * args.steps / (ms_dev / 1e3), ms_per_step=ms_dev / args.steps, clocks=clocks,
               e2e=dict(value=tokens_per_step * args.steps / (ms_e2e / 1e3), unit="tokens/s",
                        h2d_bytes_per_step=int(tmpl_host.numel() * 8), d2h_bytes_per_step=int(out_host.numel() * 8)),
               gpu_launches=int(n_launch / max(1, (args.steps + args.warmup))) * args.steps)
    res["roofline"] = sample_roofline(model, nb, res["ms_per_step"], args.gen_tokens)
    res["params"] = param_count(model)
    res["outputs"] = outputs
    del model
    torch.cuda.empty_cache()
    return res


def sample_roofline(model, nb, ms_per_step, gen_tokens, ctx_len=65):
    """Dominant decode kernel = decode_step_kernel (one launch per token: all layers + logits, weight streaming).
    Algorithmic bytes per launch (SURVEY §8(d)): every bf16 weight once (7.858 GB) + the K|V rows of the cached
    tokens (491,520 B x t per sequence).  Timed live with CUDA events over launches of the kernel alone at the mean
    memory length of the generation (each launch streams 7.9 GB >> the 126 MB L2, so nothing is served from cache)."""
    from cogview_b200 import ops
    from cogview_b200.mpu import kv_cache
    from cogview_b200.mpu.decode import DecodeRunner
    pk = peaks()
    tr = model.transformer
    c = kv_cache._Caches(tr, nb, torch.device("cuda"))
    c.buf.normal_()
    t_mean = ctx_len + gen_tokens // 2
    c.t = t_mean
    r = DecodeRunner(model, c, use_graph=False)
    if not r.persistent:
        # default path: one kernel per operation; the dominant kernel is linear_small_m_kernel (4 launches per layer + the
        # logits = 193 per token, every one streaming its own weight matrix: 7.86 GB per token, nothing served from L2).
        # Timed live with CUDA events over exactly those 193 launches, back to back on the current stream with the
        # programmatic-dependent-launch overlap they have inside the step.
        r._check_params()
        h = tr.hidden_size
        xs = {h: torch.randn((nb, h), device="cuda").to(torch.bfloat16), 4 * h: torch.randn((nb, 4 * h), device="cuda").to(torch.bfloat16)}
        outs = {n: torch.empty((nb, n), dtype=torch.bfloat16, device="cuda") for n in (h, 3 * h, 4 * h)}
        lg = torch.empty((nb, r.wte.shape[0]), dtype=torch.float32, device="cuda")

        def all_linears():
            for P in r.params:
                ops.linear_small_m(xs[h], P[2], P[3], out=outs[3 * h])
                ops.linear_small_m(xs[h], P[4], P[5], out=outs[h])
                ops.linear_small_m(xs[h], P[10], P[11], act=ops.ACT_GELU, out=outs[4 * h])
                ops.linear_small_m(xs[4 * h], P[12], P[13], out=outs[h])
            ops.linear_small_m(xs[h], r.wte, out=lg)
        for _ in range(3):
            all_linears()
        torch.cuda.synchronize()
        reps = 10
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            all_linears()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        n_l = 4 * len(r.params) + 1
        wbytes = sum(P[i].numel() * 2 for P in r.params for i in (2, 4, 10, 12)) + r.wte.numel() * 2
        achieved = wbytes / (ms / 1e3) / 1e9
        del r, c
        return dict(kernel="linear_small_m_kernel", bound="hbm", achieved=achieved, peak=pk["hbm"], unit="GB/s",
                    frac=achieved / pk["hbm"], traffic=measured_traffic("linear_small_m_kernel"), peak_source=pk["src"],
                    launches_per_step=n_l * gen_tokens, bytes_per_launch=wbytes / n_l, avg_launch_us=ms * 1e3 / n_l,
                    share_of_step=ms * gen_tokens / ms_per_step,
                    note="algorithmic bytes = the weight matrix of each launch (mean %.1f MB; all %d launches of a token "
                         "= 7.86 GB); timed over the %d launches of one token back to back; share_of_step = that x tokens "
                         "/ step (the rest: Sandwich-LN glue, cached attention, sampling)" % (wbytes / n_l / 1e6, n_l, n_l))
    r._check_params()
    r.ids.fill_(7)
    r.pos.fill_(t_mean)
    r.cur_len.fill_(t_mean)
    for _ in range(3):
        r._run()
    torch.cuda.synchronize()
    reps = 20
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        r._run()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    wbytes = sum(p.numel() * 2 for p in model.parameters())
    kvbytes = len(tr.layers) * nb * t_mean * 2 * tr.hidden_size * 2
    nbytes = wbytes + kvbytes
    achieved = nbytes / (ms / 1e3) / 1e9
    del r, c
    return dict(kernel="decode_step_kernel", bound="hbm", achieved=achieved, peak=pk["hbm"], unit="GB/s",
                frac=achieved / pk["hbm"], traffic=measured_traffic("decode_step_kernel"), peak_source=pk["src"],
                launches_per_step=gen_tokens, bytes_per_launch=nbytes, avg_launch_us=ms * 1e3,
                share_of_step=ms * gen_tokens / ms_per_step,
                note="bytes = all weights + K|V of t=%d cached tokens x %d seqs; share_of_step = kernel x tokens / step" % (
                    t_mean, nb))


# ----------------------------------------------------------------------------------------------------
# training workload (configs[2])
# ----------------------------------------------------------------------------------------------------
def run_train(args, cfg, world, rank, dev_index, steps, warmup):
    from cogview_b200 import mpu
    from cogview_b200.model import (PyTorchDistributedDataParallel, gpt2_get_params_for_weight_decay_optimization)
    from cogview_b200.optim import FusedAdamW
    torch.manual_seed(100 + rank)      # weights and dropout masks: the same run for the same arguments
    model = build_model(cfg, 0, "cuda", dropout=args.dropout).train()
    groups = gpt2_get_params_for_weight_decay_optimization(model)
    for g in groups:
        g.setdefault("weight_decay", 0.01)
    opt = FusedAdamW(groups, lr=4e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.01, max_grad_norm=1.0)
    net = model
    reserved = 0
    if world > 1:
        # the gradient all-reduce (pretrain_gpt2.py:99-105) runs as NCCL kernels NEXT TO the backward GEMMs: keep a few
        # SMs out of the persistent GEMM grid for them (a grid sized to all 148 SMs would find some taken and run a
        # second, nearly empty wave), and cap NCCL's CTAs to what was reserved (main() sets NCCL_MAX_CTAS).  Measured at
        # N = 2 (4 x 1088 tokens per GPU): 182.4 ms with nothing reserved (NCCL up to 32 CTAs), 183.0 ms with 16, 180.1 ms
        # with 8 (N = 1: 166.9 ms) — profiles/r02_train_2gpu_reserved_sms.txt
        from cogview_b200 import _lib
        reserved = int(os.environ.get("COGVIEW_B200_RESERVE_SMS", "8"))
        _lib.lib().cv_set_reserved_sms(reserved)
        net = PyTorchDistributedDataParallel(model, device_ids=[torch.cuda.current_device()],
                                             gradient_as_bucket_view=True, bucket_cap_mb=200)
    b, s = args.batch, cfg["max_sequence_length"] - 1
    g = torch.Generator().manual_seed(100 + rank)
    host_tokens = torch.cat((torch.randint(8192, 58192, (b, 64), generator=g),
                             torch.randint(0, 8192, (b, s + 1 - 64), generator=g)), dim=1).pin_memory()
    dev_tokens = host_tokens.cuda()
    pos = torch.arange(s, device="cuda").unsqueeze(0).expand(b, -1).contiguous()
    mask = torch.tril(torch.ones((1, 1, s, s), device="cuda"))
    loss_host = torch.zeros(1).pin_memory()
    last = {}

    def one_step(tok):
        tokens, labels = tok[:, :-1].contiguous(), tok[:, 1:].contiguous()
        logits, *_ = net(tokens, pos, mask, None, None, 0)
        losses = mpu.vocab_parallel_cross_entropy(logits, labels)
        loss = losses.mean()
        for p in model.parameters():
            p.grad = None
        loss.backward()
        opt.step()
        return loss

    def step_dev():
        last["loss"] = one_step(dev_tokens)

    def step_e2e():
        loss = one_step(host_tokens.cuda(non_blocking=True))
        loss_host.copy_(loss.detach().float().view(1), non_blocking=True)
        torch.cuda.current_stream().synchronize()

    tokens_per_step = b * s * world
    l0 = launches()
    ms_dev, clocks = timed(step_dev, steps, warmup, dev_index)
    n_launch = launches() - l0
    outputs = {}
    if args.dump_outputs:
        # the step returns the loss and updates the weights in place (the end-to-end steps below update them again)
        g = torch.Generator().manual_seed(0)
        outputs["train_loss"] = last["loss"].detach().view(1)
        outputs["train_weights_sample"] = torch.cat([
            p.detach().reshape(-1)[torch.randint(0, p.numel(), (min(p.numel(), 4096),), generator=g).cuda()].float()
            for p in model.parameters()])
    ms_e2e, _ = timed(step_e2e, steps, 1, dev_index)
    loss_val = float(last["loss"].item())
    assert loss_val == loss_val and loss_val < 20.0, "training loss is not finite"
    L, h, V = cfg["num_layers"], cfg["hidden_size"], cfg["vocab_size"]
    flops_per_token = 3 * (2 * 12 * L * h * h + 2 * h * V + 0.5 * 4 * L * s * h)   # SURVEY §8(d)
    pk = peaks()
    achieved = flops_per_token * tokens_per_step / world / (ms_dev / steps / 1e3) / 1e12
    res = dict(value=tokens_per_step * steps / (ms_dev / 1e3), unit="tokens/s", ms_per_step=ms_dev / steps,
               steps=steps, warmup=warmup, clocks=clocks, loss=loss_val,
               e2e=dict(value=tokens_per_step * steps / (ms_e2e / 1e3), unit="tokens/s",
                        h2d_bytes_per_step=int(host_tokens.numel() * 8), d2h_bytes_per_step=4),
               gpu_launches=int(n_launch / max(1, steps + warmup)) * steps,
               config=dict(workload="configs[2]: 4B training step, bf16, %d x %d tokens per GPU, dropout %.2f (embedding, "
                                    "attention, hidden), AdamW + clip 1.0, no activation recompute" % (b, s, args.dropout),
                           global_batch=b * world,
                           parallelism="dp%d" % world),
               step_flops_per_gpu=flops_per_token * tokens_per_step / world,
               roofline_step=dict(bound="tensor", achieved=achieved, peak=pk["tf_sust"], unit="TFLOP/s",
                                  frac=achieved / pk["tf_sust"], peak_source=pk["src"],
                                  note="whole step (all kernels) vs sustained cuBLAS bf16 peak"))
    res["config"]["reserved_sms_for_nccl"] = reserved
    if world > 1:
        from cogview_b200 import _lib
        _lib.lib().cv_set_reserved_sms(0)
    res["roofline"] = gemm_roofline(cfg, b * s)
    res["outputs"] = outputs
    del net, model, opt
    torch.cuda.empty_cache()
    return res


def gemm_roofline(cfg, M):
    """Dominant training kernel = gemm_kernel (tcgen05).  FLOPs per launch = 2*M*N*K; timed live with CUDA events
    over the four forward GEMM shapes of a layer, rotating through 6 weight sets (> L2)."""
    from cogview_b200 import ops
    pk = peaks()
    h = cfg["hidden_size"]
    shapes = [("qkv", 3 * h, h), ("out", h, h), ("h_to_4h", 4 * h, h), ("4h_to_h", h, 4 * h)]
    out = {}
    tot_f, tot_ms, n = 0.0, 0.0, 0
    for name, N, K in shapes:
        ws = [torch.randn((N, K), device="cuda").to(torch.bfloat16) for _ in range(6)]
        x = torch.randn((M, K), device="cuda").to(torch.bfloat16)
        for w in ws[:2]:
            ops.gemm(x, w)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(3):
            for w in ws:
                ops.gemm(x, w)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 18
        out[name] = dict(M=M, N=N, K=K, us=ms * 1e3, tflops=2.0 * M * N * K / ms / 1e9)
        tot_f += 2.0 * M * N * K
        tot_ms += ms
        n += 1
        del ws, x
    achieved = tot_f / tot_ms / 1e9
    return dict(kernel="gemm_kernel", bound="tensor", achieved=achieved, peak=pk["tf_burst"], unit="TFLOP/s",
                frac=achieved / pk["tf_burst"], traffic=measured_traffic("gemm_kernel"),
                traffic_note="ncu capture of the qkv shape (profiles/r01_traffic.json): operands read once",
                peak_source=pk["src"], shapes=out,
                flops_per_launch=tot_f / n, avg_launch_us=tot_ms * 1e3 / n)


# ----------------------------------------------------------------------------------------------------
# VQ-VAE tokenizer workload (configs[3]): encode + quantise + decode of 256x256 images
# ----------------------------------------------------------------------------------------------------
def run_vqvae(args, world, rank, dev_index, steps, warmup):
    from cogview_b200 import recipes, vqvae
    model = vqvae.new_model()
    model.load_state_dict(recipes.vqvae_state_dict(seed=0))
    model = model.cuda().eval()
    B = args.vq_batch
    g = torch.Generator().manual_seed(rank)
    host_img = torch.randn((B, 3, 256, 256), generator=g).pin_memory()
    dev_img = host_img.cuda()
    host_out = torch.empty((B, 3, 256, 256)).pin_memory()
    keep = {}

    def step_dev():
        codes = vqvae.img2code(model, dev_img)
        keep["codes"] = codes
        keep["rec"] = vqvae.code2img(model, codes.view(B, 32, 32))

    def step_e2e():
        img = host_img.cuda(non_blocking=True)
        codes = vqvae.img2code(model, img)
        rec = vqvae.code2img(model, codes.view(B, 32, 32))
        host_out.copy_(rec, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    l0 = launches()
    ms_dev, clocks = timed(step_dev, steps, warmup, dev_index)
    n_launch = launches() - l0
    outputs = {}
    if args.dump_outputs:
        rec = keep["rec"].reshape(-1)
        idx = torch.randperm(rec.numel(), generator=torch.Generator().manual_seed(0))[:1 << 22].sort().values
        outputs = dict(vqvae_codes=keep["codes"], vqvae_images_sample=rec[idx.cuda()])
    ms_e2e, _ = timed(step_e2e, steps, 1, dev_index)
    assert keep["codes"].shape == (B, 1024) and int(keep["codes"].max()) < 8192
    assert bool(torch.isfinite(keep["rec"]).all())
    imgs = B * world
    gflop_per_image = 44.0 + 4.29 + 176.3            # SURVEY §8(d): encoder + distance + decoder
    pk = peaks()
    achieved = gflop_per_image * imgs / world / (ms_dev / steps / 1e3) / 1e3
    res = dict(value=imgs * steps / (ms_dev / 1e3), unit="images/s", code_tokens_per_s=imgs * 1024 * steps / (ms_dev / 1e3),
               ms_per_step=ms_dev / steps, steps=steps, warmup=warmup, clocks=clocks,
               e2e=dict(value=imgs * steps / (ms_e2e / 1e3), unit="images/s",
                        h2d_bytes_per_step=int(host_img.numel() * 4), d2h_bytes_per_step=int(host_out.numel() * 4)),
               gpu_launches=int(n_launch / max(1, steps + warmup)) * steps,
               config=dict(workload="configs[3]: VQ-VAE (new_model(): 512 ch, 8192 codes) img2code + code2img, %d "
                                    "synthetic 256x256 images per GPU, bf16 tensor-core convs, fp32-rescored arg-min" % B,
                           parallelism="dp%d (independent images per rank, no collective)" % world),
               roofline_step=dict(bound="tensor", achieved=achieved, peak=pk["tf_sust"], unit="TFLOP/s",
                                  frac=achieved / pk["tf_sust"], peak_source=pk["src"],
                                  note="whole round trip (224.6 GFLOP/image algorithmic) vs sustained cuBLAS bf16 peak"),
               outputs=outputs)
    del model
    torch.cuda.empty_cache()
    return res


def usable_cores():
    """Host cores this process may actually use: affinity mask and cgroup CPU quota, not the machine's core count."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(int(txt[0]) / int(txt[1]))))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, q // per))
        except (OSError, ValueError, IndexError):
            pass
    return n


_CPU_THREADS = None


def best_cpu_threads():
    """The CPU arm gets its best shot: the thread count (<= usable cores) with the highest measured throughput on a
    layer-sized fp32 GEMM — on many-core hosts the full count is often slower than a fraction of it."""
    global _CPU_THREADS
    if _CPU_THREADS is not None:
        torch.set_num_threads(_CPU_THREADS)
        return _CPU_THREADS
    top = usable_cores()
    cands = sorted({c for c in (top, top // 2, top // 4, 64, 32, 16, 8) if 1 <= c <= top}, reverse=True)
    a, b = torch.randn((1088, 2560)), torch.randn((2560, 2560))
    best, best_t = top, float("inf")
    for c in cands:
        torch.set_num_threads(c)
        torch.mm(a, b)
        t0 = time.perf_counter()
        for _ in range(3):
            torch.mm(a, b)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
    _CPU_THREADS = best
    torch.set_num_threads(best)
    return best


def cpu_baseline_vqvae(nimg=4):
    if reference_available() and os.environ.get("COGVIEW_B200_CPU_ARM", "reference") != "port":
        from cogview_b200 import recipes
        from oracle import ref_harness
        R = ref_harness.load()
        cores = best_cpu_threads()
        model = R["vq_api"].new_model()
        model.load_state_dict(recipes.vqvae_state_dict(seed=0))
        model.eval()
        img = recipes.images(nimg, size=256, seed=1)
        with torch.no_grad():
            t0 = time.perf_counter()
            codes = R["vq_api"].img2code(model, img)
            R["vq_api"].code2img(model, codes.view(nimg, 32, 32))
            dt = time.perf_counter() - t0
        return dict(value=nimg / dt, unit="images/s", cores=cores, kind="reference",
                    sample="reference vqvae.api (unmodified, oracle/_ref), fp32, %d threads: img2code + code2img of %d "
                           "256x256 images (%.1f s)" % (cores, nimg, dt))
    from oracle import cogview_oracle as O
    from oracle import recipes
    cores = best_cpu_threads()
    sd = recipes.vqvae_state_dict(seed=0)
    img = recipes.images(nimg, size=256, seed=1)
    t0 = time.perf_counter()
    codes = O.img2code(sd, img)
    O.code2img(sd, codes.view(nimg, 32, 32))
    dt = time.perf_counter() - t0
    return dict(value=nimg / dt, unit="images/s", cores=cores, kind="port",
                sample="oracle port, fp32, %d threads (best of the calibrated counts): img2code + code2img of %d 256x256 images (%.1f s)" % (cores, nimg, dt))


# ----------------------------------------------------------------------------------------------------
# CPU baseline: the oracle port of the reference path on the host cores
# ----------------------------------------------------------------------------------------------------
def reference_available():
    try:
        from oracle import ref_harness
        return ref_harness.available()
    except Exception:
        return False


def cpu_reference_sample(cfg, nb, gen_tokens, budget_s=20.0):
    """The reference's OWN modules (oracle/_ref or /root/reference: model/gpt2_modeling.py GPT2Model over
    mpu/sparse_transformer.py, unmodified, under the four harness shims) on the host cores, fp32: the decode call of
    generation/sampling.py:147-151 — one new token per beam, hidden-state `mems` of length t, so the whole memory is
    re-normalised and re-projected every step (mpu/sparse_transformer.py:320,136-141).  Bounded sample: a
    2-layer 4B-width model (embedding + logits included) timed at a few memory lengths; per-layer cost fitted
    linearly in t and integrated over the generated positions x 48 layers + the per-step head cost."""
    from oracle import ref_harness
    R = ref_harness.load()
    cores = best_cpu_threads()
    NL = 2
    h, heads, V = cfg["hidden_size"], cfg["num_attention_heads"], cfg["vocab_size"]
    t_start = time.perf_counter()
    torch.manual_seed(0)
    model = R["gpt2_modeling"].GPT2Model(
        num_layers=NL, vocab_size=V, hidden_size=h, num_attention_heads=heads, embedding_dropout_prob=0.0,
        attention_dropout_prob=0.0, output_dropout_prob=0.0, max_sequence_length=cfg["max_sequence_length"],
        max_memory_length=cfg["max_sequence_length"], checkpoint_activations=False).eval()
    pts = []
    with torch.no_grad():
        tok = torch.randint(0, 8192, (nb, 1))
        # head cost: embedding + final LayerNorm + logits GEMM of one token (a 0-layer pass is not constructible)
        x = torch.randn((nb, 1, h))
        t0 = time.perf_counter()
        for _ in range(3):
            torch.nn.functional.linear(model.transformer.final_layernorm(x), model.word_embeddings.weight)
        head_s = (time.perf_counter() - t0) / 3
        for t in (64, 576, 1088):
            mems = [torch.randn((nb, t, h)) for _ in range(NL + 1)]
            pos = torch.full((nb, 1), t, dtype=torch.long)
            model(tok, pos, 0, None, None, 0, *mems)                       # warm-up
            t0 = time.perf_counter()
            reps = 0
            while reps < 2 or (time.perf_counter() - t0 < 2.0 and reps < 50):
                model(tok, pos, 0, None, None, 0, *mems)
                reps += 1
            pts.append((t, (time.perf_counter() - t0) / reps))
            if time.perf_counter() - t_start > budget_s:
                break
    per_layer = [(t, max(0.0, c - head_s) / NL) for t, c in pts]
    n = len(per_layer)
    mt, mc = sum(q[0] for q in per_layer) / n, sum(q[1] for q in per_layer) / n
    bcoef = (sum((q[0] - mt) * (q[1] - mc) for q in per_layer) / max(1e-12, sum((q[0] - mt) ** 2 for q in per_layer))
             if n > 1 else 0.0)
    acoef = mc - bcoef * mt
    ctx = 65
    total = sum(cfg["num_layers"] * (acoef + bcoef * t) + head_s for t in range(ctx, ctx + gen_tokens))
    wall = time.perf_counter() - t_start
    return dict(value=nb * gen_tokens / total, unit="tokens/s", cores=cores, kind="reference", sample_wall_s=wall,
                sample="reference GPT2Model (unmodified, oracle/_ref), fp32, %d threads: %d-layer 4B-width model, one decode "
                       "call per memory length %s (batch %d, hidden-state mems); per-layer cost fitted linearly, x %d "
                       "layers + head, integrated over %d positions (= %.0f s per full step); %.1f s of CPU work" % (
                           cores, NL, [q[0] for q in pts], nb, cfg["num_layers"], gen_tokens, total, wall))


def cpu_baseline_sample(cfg, nb, gen_tokens, budget_s=20.0):
    if reference_available() and os.environ.get("COGVIEW_B200_CPU_ARM", "reference") != "port":
        return cpu_reference_sample(cfg, nb, gen_tokens, budget_s)
    return cpu_port_sample(cfg, nb, gen_tokens, budget_s)


def cpu_port_sample(cfg, nb, gen_tokens, budget_s=20.0):
    """Reference semantics (generation/sampling.py:147-151 over mpu/sparse_transformer.py:320,136-141): each step
    re-normalises and re-projects the whole hidden-state memory.  Sample: ONE 4B-shaped layer (fp32) timed at a
    few memory lengths with batch nb, cost fitted linearly in the memory length and integrated over the
    generated positions x num_layers, plus the last-token logits GEMM per step."""
    from oracle import cogview_oracle as O
    from oracle import recipes
    cores = best_cpu_threads()
    one = dict(cfg)
    one["num_layers"] = 1
    sd = recipes.gpt2_state_dict(seed=1, perturb=False, **one)
    sd = {k: v for k, v in sd.items()}
    heads = cfg["num_attention_heads"]
    h = cfg["hidden_size"]
    pts = []
    t_start = time.perf_counter()
    with torch.no_grad():
        for t in (64, 320, 576, 832, 1088):
            mem = torch.randn((nb, t, h))
            x = torch.randn((nb, 1, h))
            mask = O.build_sep_mask(1, t + 1, 0)
            t0 = time.perf_counter()
            O.transformer_layer(sd, 0, x, mask, heads, mem=mem)
            once = time.perf_counter() - t0
            reps = int(min(50, max(2, 2.0 / max(once, 1e-3))))      # ~2 s of CPU work per memory length
            t0 = time.perf_counter()
            for _ in range(reps):
                O.transformer_layer(sd, 0, x, mask, heads, mem=mem)
            pts.append((t, (time.perf_counter() - t0) / reps))
            if time.perf_counter() - t_start > budget_s:
                break
        xl = torch.randn((nb, h))
        t0 = time.perf_counter()
        torch.nn.functional.linear(xl, sd["word_embeddings.weight"])
        logits_s = time.perf_counter() - t0
    # least-squares line  cost(t) = a + b t
    n = len(pts)
    mt, mc = sum(p[0] for p in pts) / n, sum(p[1] for p in pts) / n
    bcoef = sum((p[0] - mt) * (p[1] - mc) for p in pts) / max(1e-12, sum((p[0] - mt) ** 2 for p in pts)) if n > 1 else 0.0
    acoef = mc - bcoef * mt
    ctx = 65
    total = sum(cfg["num_layers"] * (acoef + bcoef * t) + logits_s for t in range(ctx, ctx + gen_tokens))
    return dict(value=nb * gen_tokens / total, unit="tokens/s", cores=cores, kind="port",
                sample="oracle port, fp32, %d threads (best of the calibrated counts): 1 of %d layers at memory lengths %s (batch %d), linear fit "
                       "integrated over %d generated positions + logits GEMM per step; %.1f s of CPU work" % (
                           cores, cfg["num_layers"], [p[0] for p in pts], nb, gen_tokens,
                           time.perf_counter() - t_start))


def cpu_reference_train(cfg):
    """The reference's GPT2Model (1 layer, 4B width) + mpu.vocab_parallel_cross_entropy, forward + backward at b=1,
    s=1088, fp32 on the host cores; per-layer cost = total - head (embedding, logits GEMM, cross-entropy), x 48."""
    from oracle import ref_harness
    R = ref_harness.load()
    cores = best_cpu_threads()
    s_len = cfg["max_sequence_length"] - 1
    h, V = cfg["hidden_size"], cfg["vocab_size"]
    torch.manual_seed(0)
    model = R["gpt2_modeling"].GPT2Model(
        num_layers=1, vocab_size=V, hidden_size=h, num_attention_heads=cfg["num_attention_heads"],
        embedding_dropout_prob=0.0, attention_dropout_prob=0.0, output_dropout_prob=0.0,
        max_sequence_length=cfg["max_sequence_length"], max_memory_length=0, checkpoint_activations=False).train()
    tok = torch.randint(0, V, (1, s_len))
    lab = torch.randint(0, V, (1, s_len))
    pos = torch.arange(s_len).unsqueeze(0)
    mask = torch.tril(torch.ones((1, 1, s_len, s_len)))
    t0 = time.perf_counter()
    logits, *_ = model(tok, pos, mask, None, None, 0)
    R["mpu"].vocab_parallel_cross_entropy(logits.contiguous().float(), lab).mean().backward()
    full_s = time.perf_counter() - t0
    hid = torch.randn((1, s_len, h), requires_grad=True)
    w = model.word_embeddings.weight
    t0 = time.perf_counter()
    lg = torch.nn.functional.linear(hid, w)
    R["mpu"].vocab_parallel_cross_entropy(lg.contiguous().float(), lab).mean().backward()
    head_s = time.perf_counter() - t0
    layer_s = max(1e-6, full_s - head_s)
    total = cfg["num_layers"] * layer_s + head_s
    return dict(value=s_len / total, unit="tokens/s", cores=cores, kind="reference",
                sample="reference GPT2Model (unmodified, oracle/_ref), fp32, %d threads: 1-layer 4B-width fwd+bwd at b=1, "
                       "s=%d (%.1f s, of which head %.1f s) -> x %d layers + head; extrapolated, optimizer not included" % (
                           cores, s_len, full_s, head_s, cfg["num_layers"]))


def cpu_baseline_train(cfg, budget_s=25.0):
    if reference_available() and os.environ.get("COGVIEW_B200_CPU_ARM", "reference") != "port":
        return cpu_reference_train(cfg)
    from oracle import cogview_oracle as O
    from oracle import recipes
    cores = best_cpu_threads()
    one = dict(cfg)
    one["num_layers"] = 1
    sd = {k: v.requires_grad_(True) for k, v in recipes.gpt2_state_dict(seed=1, perturb=False, **one).items()}
    s = cfg["max_sequence_length"] - 1
    h = cfg["hidden_size"]
    x = torch.randn((1, s, h), requires_grad=True)
    mask = torch.tril(torch.ones((1, 1, s, s)))
    t0 = time.perf_counter()
    y = O.transformer_layer(sd, 0, x, mask, cfg["num_attention_heads"])
    y.sum().backward()
    layer_s = time.perf_counter() - t0
    t0 = time.perf_counter()
    hid = torch.randn((s, h), requires_grad=True)
    logits = torch.nn.functional.linear(hid, sd["word_embeddings.weight"])
    O.vocab_parallel_cross_entropy(logits, torch.randint(0, cfg["vocab_size"], (s,))).mean().backward()
    head_s = time.perf_counter() - t0
    total = cfg["num_layers"] * layer_s + head_s
    return dict(value=s / total, unit="tokens/s", cores=cores, kind="port",
                sample="oracle port, fp32, %d threads (best of the calibrated counts): 1 of %d layers fwd+bwd at b=1, s=%d (%.1f s) x %d + logits/CE "
                       "fwd+bwd (%.1f s); extrapolated, optimizer not included" % (cores, cfg["num_layers"], s, layer_s,
                                                                                  cfg["num_layers"], head_s))


# ----------------------------------------------------------------------------------------------------
def write_outputs(directory, outputs):
    """One DIR/<name>.npy per output, as float32 (exact for the token ids and codes, which stay below 2**24)."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, t in outputs.items():
        np.save(os.path.join(directory, name + ".npy"), t.detach().float().cpu().numpy())


def _compact(d, keys):
    return {k: d[k] for k in keys if k in d}


def main():
    args = parse()
    cfg = MODEL_4B if args.model == "4b" else MODEL_TINY
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    workload_name = ("configs[1]: CogView-base 4B (48L, d=2560, 40H, V=58240), seq 1089, bf16, AR sampling: prefill 65 "
                     "+ generate %d tokens, %d beams/GPU, top-k 200; weight-streaming decode kernels + one sampling "
                     "kernel, one CUDA-graph replay per token" % (args.gen_tokens, args.batch))
    # BASELINE.json's metric; `value` is the AR-sampling tokens/s (configs[1]), the training step (configs[2]) and the
    # VQ-VAE round trip (configs[3]) are summarised in config.train / config.vqvae and in full in `train` / `vqvae`
    base = dict(metric="tokens/sec (train + AR sample) CogView-4B seq1089 @1/2/4/8 B200; %roofline", unit="tokens/s",
                n_gpus=world, steps=args.steps, warmup=args.warmup, higher_is_better=True, scaling="weak",
                vs_baseline=None, dtype="bf16", data="synthetic tokens, random-init weights")

    if args.impl == "reference":
        # The reference's own CPU path on this box's host cores.  A "step" here is one bounded sample of the workload
        # (see cpu_reference_sample); ms_per_step is the sample's real duration, value the throughput it implies.
        if rank != 0:
            return
        t0 = time.perf_counter()
        vals, walls = [], []
        for _ in range(args.warmup and 1):
            cpu_baseline_sample(cfg, args.batch, args.gen_tokens, budget_s=8.0)
        for _ in range(args.steps):
            ts = time.perf_counter()
            cb = cpu_baseline_sample(cfg, args.batch, args.gen_tokens, budget_s=15.0)
            walls.append(time.perf_counter() - ts)
            vals.append(cb["value"])
        cb["value"] = statistics.median(vals)
        line = dict(base, impl="reference", value=cb["value"], ms_per_step=statistics.median(walls) * 1e3,
                    steps=len(vals), dtype="f32", cpu_baseline=cb,
                    config=dict(workload=workload_name, global_batch=args.batch, seq_len=1089, parallelism="cpu",
                                note="each step = one bounded sample of the workload on the host cores"),
                    e2e=dict(value=cb["value"], unit="tokens/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                    gpu_launches=0, wall_s=time.perf_counter() - t0)
        if args.workload in ("train", "both", "all"):
            tb = cpu_baseline_train(cfg)
            line["config"]["train"] = dict(value=tb["value"], unit="tokens/s", kind=tb["kind"], cores=tb["cores"])
        print(json.dumps(line))
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU: the product path has no CPU fallback (use --impl reference for the "
                         "CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_MAX_CTAS", os.environ.get("COGVIEW_B200_RESERVE_SMS", "8"))
        torch.distributed.init_process_group("nccl")
        from cogview_b200 import mpu
        mpu.initialize_model_parallel(1)

    line = dict(base)
    outputs = {}
    if args.workload in ("sample", "both", "all"):
        r = run_sample(args, cfg, world, rank, local_rank)
        outputs.update(r.pop("outputs"))
        line.update(value=r["value"], ms_per_step=r["ms_per_step"], e2e=r["e2e"], clocks=r["clocks"],
                    gpu_launches=r["gpu_launches"], roofline=r["roofline"],
                    config=dict(workload=workload_name, global_batch=args.batch * world, seq_len=1089,
                                parallelism="dp%d (independent sequences per rank, no collective)" % world,
                                l2="each decode step streams 7.9 GB of weights (>> 126 MB L2)", params=r["params"]))
    if args.workload in ("vqvae", "all"):
        v = run_vqvae(args, world, rank, local_rank, args.steps, max(3, args.warmup))
        outputs.update(v.pop("outputs"))
        if args.workload == "vqvae":
            line.update(metric="images/sec (VQ-VAE encode+quantise+decode, 256x256)", unit="images/s", value=v["value"],
                        ms_per_step=v["ms_per_step"], e2e=v["e2e"], clocks=v["clocks"], gpu_launches=v["gpu_launches"],
                        roofline=v["roofline_step"], config=v["config"], steps=v["steps"], warmup=v["warmup"])
        else:
            line["config"]["vqvae"] = dict(value=v["value"], unit="images/s", ms_per_step=v["ms_per_step"],
                                           frac_of_sustained_tensor_peak=v["roofline_step"]["frac"])
        line["vqvae"] = v
    if args.workload in ("train", "both", "all"):
        tsteps = args.train_steps or args.steps
        t = run_train(args, cfg, world, rank, local_rank, tsteps, max(3, args.warmup))
        outputs.update(t.pop("outputs"))
        if args.workload == "train":
            line.update(metric="tokens/sec (train) CogView-4B seq1089", value=t["value"], ms_per_step=t["ms_per_step"],
                        e2e=t["e2e"], clocks=t["clocks"], gpu_launches=t["gpu_launches"], roofline=t["roofline"],
                        config=t["config"], steps=t["steps"], warmup=t["warmup"])
        else:
            # configs[2] — the workload with the one collective of the path (bf16 gradient all-reduce): kept inside
            # `config` so that the per-N records of a scaling run carry it
            line["config"]["train"] = dict(value=t["value"], unit="tokens/s", ms_per_step=t["ms_per_step"],
                                           global_batch=t["config"]["global_batch"], e2e=t["e2e"]["value"],
                                           step_frac_of_sustained_tensor_peak=t["roofline_step"]["frac"],
                                           gemm_frac_of_burst_peak=t["roofline"]["frac"], loss=t["loss"],
                                           exposed_comm_ms=t.get("exposed_comm_ms"))
        line["train"] = t
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, outputs)
    if rank == 0 and (args.skip_cpu_baseline or world > 1):
        # the CPU baseline is reported at N = 1 only (--skip-cpu-baseline: development runs)
        line["cpu_baseline"] = None
        print(json.dumps(line))
    elif rank == 0:
        if args.workload in ("sample", "both", "all"):
            line["cpu_baseline"] = cpu_baseline_sample(cfg, args.batch, args.gen_tokens)
        if args.workload in ("vqvae", "all"):
            line["vqvae"]["cpu_baseline"] = cpu_baseline_vqvae()
            if args.workload == "vqvae":
                line["cpu_baseline"] = line["vqvae"]["cpu_baseline"]
        if args.workload in ("train", "both", "all"):
            line["train"]["cpu_baseline"] = cpu_baseline_train(cfg)
            if args.workload == "train":
                line["cpu_baseline"] = line["train"]["cpu_baseline"]
        print(json.dumps(line))
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
