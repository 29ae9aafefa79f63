"""Thin functional wrappers over the C ABI: allocate outputs with torch, pass raw pointers + stream.

These are the only places that call into libcogview_b200.so; the `mpu` / `model` / `vqvae` mirrors of the
reference interface are built on them.
"""
import torch

from . import _lib
from ._lib import check, lib, ptr, require_cuda, stream_ptr

ACT_NONE = 0
ACT_GELU = 1
ACT_RELU = 2
ACT_GELU_GRAD = 3   # multiply the result by gelu'(aux) (GELU backward fused into the dgrad GEMM)


def gemm(a, b, *, a_mn_major=False, b_mn_major=False, bias=None, act=ACT_NONE, out_dtype=torch.bfloat16,
         absmax=None, want_preact=False, out=None, block_n=0, aux=None, dropout=None):
    """C[M,N] = op(A)[M,K] @ op(B)[N,K]^T (+bias) (+GELU).

    a: [M,K] (or [K,M] when a_mn_major); b: [N,K] (or [K,N] when b_mn_major); both bf16, last dim contiguous.
    absmax: optional 1-element fp32 tensor updated with atomic max |C|.
    Returns C, or (C, preact) when want_preact.
    """
    require_cuda(a, b, bias, absmax)
    assert a.dtype == torch.bfloat16 and b.dtype == torch.bfloat16
    assert a.dim() == 2 and b.dim() == 2 and a.stride(1) == 1 and b.stride(1) == 1
    if a_mn_major:
        K, M = a.shape
    else:
        M, K = a.shape
    if b_mn_major:
        Kb, N = b.shape
    else:
        N, Kb = b.shape
    assert K == Kb, "inner dimensions differ: %d vs %d" % (K, Kb)
    if out is None:
        out = torch.empty((M, N), dtype=out_dtype, device=a.device)
    assert out.stride(1) == 1
    pre = torch.empty((M, N), dtype=torch.bfloat16, device=a.device) if want_preact else None
    if act == ACT_GELU_GRAD:
        assert aux is not None and aux.shape == (M, N) and aux.dtype == torch.bfloat16 and not want_preact
        assert aux.stride(1) == 1 and aux.stride(0) == out.stride(0)
        pre = aux
    if bias is not None:
        assert bias.dtype == torch.bfloat16 and bias.numel() == N
    if dropout is not None and dropout[0] > 0:
        rc = lib().cv_gemm_bf16_dropout(ptr(a), int(a_mn_major), a.stride(0), ptr(b), int(b_mn_major), b.stride(0),
                                        ptr(out), int(out.dtype == torch.float32), out.stride(0), ptr(pre), ptr(bias),
                                        int(act), ptr(absmax), M, N, K, block_n, float(dropout[0]), int(dropout[1]),
                                        int(dropout[2]), stream_ptr())
    else:
        rc = lib().cv_gemm_bf16(ptr(a), int(a_mn_major), a.stride(0), ptr(b), int(b_mn_major), b.stride(0),
                                ptr(out), int(out.dtype == torch.float32), out.stride(0), ptr(pre), ptr(bias), int(act),
                                ptr(absmax), M, N, K, block_n, stream_ptr())
    check(rc, "cv_gemm_bf16")
    return (out, pre) if want_preact else out


# ----------------------------------------------------------------------------------------------------
# abs-max LayerNorm
# ----------------------------------------------------------------------------------------------------
def new_scalars(n, device):
    """n zero-initialised fp32 scalars (abs-max accumulators must start at a non-negative value)."""
    return torch.zeros(n, dtype=torch.float32, device=device)


def absmax(x, out=None):
    require_cuda(x)
    x = x.contiguous()
    if out is None:
        out = torch.zeros(1, dtype=torch.float32, device=x.device)
    assert x.dtype in (torch.float32, torch.bfloat16)
    check(lib().cv_absmax(ptr(x), int(x.dtype == torch.bfloat16), x.numel(), ptr(out), stream_ptr()), "cv_absmax")
    return out


def layernorm_absmax_fwd(x, absmax_in, gamma, beta, eps, *, residual=None, out_dtype=torch.bfloat16,
                         absmax_out=None, save_stats=False):
    """x: [rows, cols] fp32|bf16 contiguous.  Returns (out, mean, rstd) (stats None unless save_stats)."""
    require_cuda(x, absmax_in, gamma, beta, residual)
    assert x.is_contiguous() and x.dim() == 2
    rows, cols = x.shape
    assert gamma.dtype == torch.bfloat16 and beta.dtype == torch.bfloat16
    out = torch.empty((rows, cols), dtype=out_dtype, device=x.device)
    mean = rstd = None
    if save_stats:
        mean = torch.empty(rows, dtype=torch.float32, device=x.device)
        rstd = torch.empty(rows, dtype=torch.float32, device=x.device)
    if residual is not None:
        assert residual.dtype == torch.float32 and residual.is_contiguous() and residual.shape == x.shape
    rc = lib().cv_layernorm_absmax_fwd(ptr(x), int(x.dtype == torch.bfloat16), ptr(absmax_in), ptr(gamma), ptr(beta),
                                       float(eps), ptr(residual), ptr(out), int(out_dtype == torch.bfloat16),
                                       ptr(absmax_out), ptr(mean), ptr(rstd), rows, cols, stream_ptr())
    check(rc, "cv_layernorm_absmax_fwd")
    return out, mean, rstd


def _drop3(dropout):
    if dropout is None or dropout[0] <= 0:
        return 0.0, 0, 0
    return float(dropout[0]), int(dropout[1]), int(dropout[2])


def dropout_mask(n, p, seed, site, device="cuda"):
    """Keep mask (uint8) of the first n elements of dropout site (seed, site) — what every fused dropout uses."""
    out = torch.empty(n, dtype=torch.uint8, device=device)
    check(lib().cv_dropout_mask(ptr(out), n, float(p), int(seed), int(site), stream_ptr()), "cv_dropout_mask")
    return out


def layernorm_absmax_bwd(x, dy, mean, rstd, gamma, *, dres=None, dx_dtype=torch.float32, dropout=None,
                         want_dxsum=False):
    """Returns (dx, dgamma, dbeta) [+ column sums of dx when want_dxsum (hidden size % 256 == 0)]."""
    require_cuda(x, dy, mean, rstd, gamma, dres)
    assert x.is_contiguous() and dy.is_contiguous()
    rows, cols = x.shape
    dx = torch.empty((rows, cols), dtype=dx_dtype, device=x.device)
    dgamma = torch.empty(cols, dtype=torch.bfloat16, device=x.device)
    dbeta = torch.empty(cols, dtype=torch.bfloat16, device=x.device)
    ws = torch.empty(lib().cv_layernorm_bwd_workspace_bytes(rows, cols) // 4, dtype=torch.float32, device=x.device)
    dxsum = torch.empty(cols, dtype=torch.bfloat16, device=x.device) if want_dxsum else None
    if dres is not None:
        assert dres.dtype == torch.float32 and dres.is_contiguous()
    rc = lib().cv_layernorm_absmax_bwd(ptr(x), int(x.dtype == torch.bfloat16), ptr(dy),
                                       int(dy.dtype == torch.bfloat16), ptr(mean), ptr(rstd), ptr(gamma), ptr(dres),
                                       ptr(dx), int(dx_dtype == torch.bfloat16), ptr(dgamma), ptr(dbeta), ptr(ws),
                                       rows, cols, *_drop3(dropout), ptr(dxsum), stream_ptr())
    check(rc, "cv_layernorm_absmax_bwd")
    if want_dxsum:
        return dx, dgamma, dbeta, dxsum
    return dx, dgamma, dbeta


# ----------------------------------------------------------------------------------------------------
# attention
# ----------------------------------------------------------------------------------------------------
def attn_fwd(q, k, v, heads, *, sep=0, want_lse=False, dropout=None):
    """q: [b, sq, heads*64] view, k/v: [b, sk, heads*64] views (last dim contiguous, bf16).
    Returns ctx [b, sq, heads*64] bf16 (and lse [b, heads, sq] fp32; and the keep-bit tensor when dropout is on)."""
    require_cuda(q, k, v)
    b, sq, hq = q.shape
    sk = k.shape[1]
    assert q.stride(2) == 1 and k.stride(2) == 1 and v.stride(2) == 1
    assert hq == heads * 64 and k.shape[2] == hq and v.shape == k.shape
    out = torch.empty((b, sq, hq), dtype=torch.bfloat16, device=q.device)
    lse = torch.empty((b, heads, sq), dtype=torch.float32, device=q.device) if want_lse else None
    dp, dseed, dsite = _drop3(dropout)
    mask = None
    if dp > 0:
        # keep bits in two layouts: [0] key-major [b, heads, key (padded to 128), query block, 4 x 32 queries] for the
        # backward, [1] query-major [b, heads, query (padded), key block, 4 x 32 keys] for the forward kernel
        mask = torch.empty((2, b, heads, ((sk + 127) // 128) * ((sq + 127) // 128) * 128, 4), dtype=torch.int32,
                           device=q.device)
    rc = lib().cv_attn_fwd(ptr(q), q.stride(1), q.stride(0), ptr(k), k.stride(1), k.stride(0), ptr(v), v.stride(1),
                           v.stride(0), ptr(out), out.stride(1), out.stride(0), ptr(lse), b, heads, 64, sq, sk,
                           int(sep), dp, dseed, dsite, ptr(mask), stream_ptr())
    check(rc, "cv_attn_fwd")
    if dp > 0:
        return (out, lse, mask) if want_lse else (out, mask)
    return (out, lse) if want_lse else out


def attn_bwd(q, k, v, out, d_out, lse, heads, *, sep=0, dropout_p=0.0, drop_mask=None):
    """Backward of attn_fwd for sq == sk.  Returns dqkv [b, s, 3*heads*64] bf16 (dQ | dK | dV)."""
    require_cuda(q, k, v, out, d_out, lse)
    b, s, h = q.shape
    assert k.shape[1] == s, "attention backward needs sq == sk"
    assert out.is_contiguous() and d_out.is_contiguous() and d_out.dtype == torch.bfloat16
    dqkv = torch.empty((b, s, 3 * h), dtype=torch.bfloat16, device=q.device)
    ws = torch.empty(lib().cv_attn_bwd_workspace_bytes(b, heads, 64, s) // 4, dtype=torch.float32, device=q.device)
    rc = lib().cv_attn_bwd(ptr(q), q.stride(1), q.stride(0), ptr(k), k.stride(1), k.stride(0), ptr(v), v.stride(1),
                           v.stride(0), ptr(out), ptr(d_out), ptr(lse), ptr(dqkv), ptr(ws), b, heads, 64, s, int(sep),
                           float(dropout_p), ptr(drop_mask), stream_ptr())
    check(rc, "cv_attn_bwd")
    return dqkv


def attn_sparse_fwd(q, k, v, heads, pivot_idx, query_window, key_window_times, *, want_lse=False, dropout=None):
    """Sparse TRAINING attention (mpu/sparse_transformer.py:675-725): q, k, v [b, s, heads*64] bf16 views,
    pivot_idx int64 [b, n_piv].  dropout: None or (p, seed, site) — dropout on the joint softmax probabilities.
    Returns ctx [b, s, heads*64] bf16 (and lse [b, heads, s] fp32; and the keep-bit tensor when dropout is on)."""
    require_cuda(q, k, v, pivot_idx)
    b, s, h = q.shape
    n_piv = pivot_idx.shape[1]
    assert q.stride(2) == 1 and k.stride(2) == 1 and v.stride(2) == 1 and h == heads * 64
    assert pivot_idx.dtype == torch.int64 and pivot_idx.shape[0] == b
    pivot_idx = pivot_idx.contiguous()
    out = torch.empty((b, s, h), dtype=torch.bfloat16, device=q.device)
    lse = torch.empty((b, heads, s), dtype=torch.float32, device=q.device) if want_lse else None
    ws = torch.empty(lib().cv_attn_sparse_workspace_bytes(b, heads, 64, n_piv), dtype=torch.uint8, device=q.device)
    dp, dseed, dsite = _drop3(dropout)
    if dp > 0:
        # keep bits in three regions (include/cogview_b200.h): band key-major, pivot key-major, query-major
        words = lib().cv_attn_sparse_drop_mask_words(b, heads, s, n_piv, int(query_window), int(key_window_times))
        mask = torch.empty(words, dtype=torch.int32, device=q.device)
        rc = lib().cv_attn_sparse_dropout_fwd(ptr(q), q.stride(1), q.stride(0), ptr(k), k.stride(1), k.stride(0), ptr(v),
                                              v.stride(1), v.stride(0), ptr(pivot_idx), ptr(out), out.stride(1),
                                              out.stride(0), ptr(lse), ptr(ws), b, heads, 64, s, n_piv,
                                              int(query_window), int(key_window_times), dp, dseed, dsite, ptr(mask),
                                              stream_ptr())
        check(rc, "cv_attn_sparse_dropout_fwd")
        return (out, lse, mask) if want_lse else (out, mask)
    rc = lib().cv_attn_sparse_fwd(ptr(q), q.stride(1), q.stride(0), ptr(k), k.stride(1), k.stride(0), ptr(v), v.stride(1),
                                  v.stride(0), ptr(pivot_idx), ptr(out), out.stride(1), out.stride(0), ptr(lse), ptr(ws),
                                  b, heads, 64, s, n_piv, int(query_window), int(key_window_times), stream_ptr())
    check(rc, "cv_attn_sparse_fwd")
    return (out, lse) if want_lse else out


def attn_sparse_bwd(q, k, v, out, d_out, lse, heads, pivot_idx, query_window, key_window_times, *, dropout_p=0.0,
                    drop_mask=None):
    """Backward of attn_sparse_fwd (dropout_p / drop_mask: the p and keep-bit tensor of a forward with dropout).
    Returns dqkv [b, s, 3*heads*64] bf16 (dQ | dK | dV)."""
    require_cuda(q, k, v, out, d_out, lse, pivot_idx)
    b, s, h = q.shape
    n_piv = pivot_idx.shape[1]
    assert out.is_contiguous() and d_out.is_contiguous() and d_out.dtype == torch.bfloat16
    pivot_idx = pivot_idx.contiguous()
    dqkv = torch.empty((b, s, 3 * h), dtype=torch.bfloat16, device=q.device)
    ws = torch.empty(lib().cv_attn_sparse_bwd_workspace_bytes(b, heads, 64, s, n_piv), dtype=torch.uint8,
                     device=q.device)
    if dropout_p > 0:
        rc = lib().cv_attn_sparse_dropout_bwd(ptr(q), q.stride(1), q.stride(0), ptr(k), k.stride(1), k.stride(0), ptr(v),
                                              v.stride(1), v.stride(0), ptr(pivot_idx), ptr(out), ptr(d_out), ptr(lse),
                                              ptr(dqkv), ptr(ws), b, heads, 64, s, n_piv, int(query_window),
                                              int(key_window_times), float(dropout_p), ptr(drop_mask), stream_ptr())
        check(rc, "cv_attn_sparse_dropout_bwd")
        return dqkv
    rc = lib().cv_attn_sparse_bwd(ptr(q), q.stride(1), q.stride(0), ptr(k), k.stride(1), k.stride(0), ptr(v), v.stride(1),
                                  v.stride(0), ptr(pivot_idx), ptr(out), ptr(d_out), ptr(lse), ptr(dqkv), ptr(ws), b,
                                  heads, 64, s, n_piv, int(query_window), int(key_window_times), stream_ptr())
    check(rc, "cv_attn_sparse_bwd")
    return dqkv


# ----------------------------------------------------------------------------------------------------
# embedding, cross-entropy, small backward helpers
# ----------------------------------------------------------------------------------------------------
def embed_fwd(ids, pos, wte, wpe, absmax_out=None, dropout=None):
    require_cuda(ids, pos, wte, wpe)
    ids = ids.contiguous().view(-1)
    pos = pos.contiguous().view(-1)
    assert ids.dtype == torch.int64 and pos.dtype == torch.int64 and ids.numel() == pos.numel()
    assert wte.dtype == torch.bfloat16 and wpe.dtype == torch.bfloat16 and wte.is_contiguous() and wpe.is_contiguous()
    h = wte.shape[1]
    out = torch.empty((ids.numel(), h), dtype=torch.float32, device=wte.device)
    check(lib().cv_embed_fwd(ptr(ids), ptr(pos), ptr(wte), ptr(wpe), ptr(out), ptr(absmax_out), ids.numel(), h,
                             *_drop3(dropout), stream_ptr()), "cv_embed_fwd")
    return out


def embed_bwd(ids, pos, dx, dwte, dwpe, dropout=None):
    """Accumulates into dwte / dwpe (bf16, contiguous)."""
    require_cuda(ids, pos, dx, dwte, dwpe)
    ids = ids.contiguous().view(-1)
    pos = pos.contiguous().view(-1)
    assert dx.dtype == torch.float32 and dx.is_contiguous()
    check(lib().cv_embed_bwd(ptr(ids), ptr(pos), ptr(dx), ptr(dwte), ptr(dwpe), ids.numel(), dwte.shape[1],
                             *_drop3(dropout), stream_ptr()), "cv_embed_bwd")


def cross_entropy_fwd(logits, target):
    """logits: [rows, V] fp32 (last dim contiguous); target int64 [rows].  Returns (loss, row_max, row_sum)."""
    require_cuda(logits, target)
    assert logits.dtype == torch.float32 and logits.dim() == 2 and logits.stride(1) == 1
    rows, V = logits.shape
    target = target.contiguous().view(-1)
    assert target.numel() == rows and target.dtype == torch.int64
    loss = torch.empty(rows, dtype=torch.float32, device=logits.device)
    rmax = torch.empty_like(loss)
    rsum = torch.empty_like(loss)
    check(lib().cv_cross_entropy_fwd(ptr(logits), logits.stride(0), ptr(target), ptr(loss), ptr(rmax), ptr(rsum), rows,
                                     V, stream_ptr()), "cv_cross_entropy_fwd")
    return loss, rmax, rsum


def cross_entropy_bwd(logits, target, rmax, rsum, grad_loss):
    require_cuda(logits, target, grad_loss)
    rows, V = logits.shape
    target = target.contiguous().view(-1)
    grad_loss = grad_loss.contiguous().view(-1).float()
    ldd = (V + 7) // 8 * 8
    dl = torch.empty((rows, ldd), dtype=torch.bfloat16, device=logits.device)
    check(lib().cv_cross_entropy_bwd(ptr(logits), logits.stride(0), ptr(target), ptr(rmax), ptr(rsum), ptr(grad_loss),
                                     ptr(dl), ldd, rows, V, stream_ptr()), "cv_cross_entropy_bwd")
    return dl[:, :V]


def gelu_bwd(pre, dact):
    require_cuda(pre, dact)
    assert pre.is_contiguous() and dact.is_contiguous() and pre.dtype == torch.bfloat16 and dact.dtype == torch.bfloat16
    out = torch.empty_like(pre)
    check(lib().cv_gelu_bwd(ptr(pre), ptr(dact), ptr(out), pre.numel(), stream_ptr()), "cv_gelu_bwd")
    return out


def colsum(dy):
    """bias gradient: sum over rows of a [rows, cols] bf16 matrix -> [cols] bf16."""
    require_cuda(dy)
    assert dy.dim() == 2 and dy.stride(1) == 1 and dy.dtype == torch.bfloat16
    rows, cols = dy.shape
    out = torch.empty(cols, dtype=torch.bfloat16, device=dy.device)
    ws = torch.empty(lib().cv_colsum_workspace_bytes(cols) // 4, dtype=torch.float32, device=dy.device)
    check(lib().cv_colsum_bf16(ptr(dy), dy.stride(0), ptr(out), ptr(ws), rows, cols, stream_ptr()), "cv_colsum_bf16")
    return out


# ----------------------------------------------------------------------------------------------------
# decode (weight-streaming) kernels
# ----------------------------------------------------------------------------------------------------
def linear_small_m(x, w, bias=None, *, act=ACT_NONE, out_dtype=torch.bfloat16, absmax=None, out=None):
    """y = x @ w^T + bias for 1 <= M <= 16 rows (x: [M,K] bf16, w: [N,K] bf16)."""
    require_cuda(x, w, bias, absmax)
    M, K = x.shape
    N = w.shape[0]
    assert x.dtype == torch.bfloat16 and w.dtype == torch.bfloat16 and x.stride(1) == 1 and w.stride(1) == 1
    if out is None:
        out = torch.empty((M, N), dtype=out_dtype, device=x.device)
    rc = lib().cv_linear_small_m(ptr(x), x.stride(0), ptr(w), w.stride(0), ptr(bias), ptr(out), out.stride(0),
                                 int(out.dtype == torch.float32), int(act), ptr(absmax), M, N, K, stream_ptr())
    check(rc, "cv_linear_small_m")
    return out


def attn_decode(qkv, cache, heads, *, cur_len=None, cur_len_dev=None, nsplit=1, out=None, workspace=None):
    """qkv: [b, 3h] bf16; cache: [b, max_len, 2h] bf16 (K|V); appends the new token at cur_len and returns
    the attention context [b, h] bf16."""
    require_cuda(qkv, cache)
    b, h3 = qkv.shape
    h = h3 // 3
    assert qkv.is_contiguous() and cache.stride(2) == 1 and cache.stride(1) == 2 * h and cache.shape[2] == 2 * h
    if out is None:
        out = torch.empty((b, h), dtype=torch.bfloat16, device=qkv.device)
    if nsplit > 1 and workspace is None:
        workspace = torch.empty(lib().cv_attn_decode_workspace_bytes(b, heads, nsplit) // 4, dtype=torch.float32,
                                device=qkv.device)
    rc = lib().cv_attn_decode(ptr(qkv), ptr(cache), cache.stride(0), ptr(cur_len_dev),
                              -1 if cur_len is None else int(cur_len), ptr(out), ptr(workspace), b, heads, 64,
                              cache.shape[1], nsplit, stream_ptr())
    check(rc, "cv_attn_decode")
    return out


def sparse_plan(is_txt, cur_len_dev, num_layers, window, num_pivot, max_sequence_length, seed_dev, idx, n_dev, err):
    """Index plan of one sparse decode step for every layer (cv_sparse_plan).  is_txt: uint8 [b, max_len]; idx: int32
    [num_layers, b, nmax] (written); n_dev, err: int32 [1]; seed_dev: int64 [1]."""
    require_cuda(is_txt, cur_len_dev, seed_dev, idx, n_dev, err)
    assert is_txt.dtype == torch.uint8 and is_txt.stride(1) == 1 and idx.dtype == torch.int32 and idx.is_contiguous()
    assert cur_len_dev.dtype == torch.int32 and n_dev.dtype == torch.int32 and seed_dev.dtype == torch.int64
    L, b, nmax = idx.shape
    assert L == num_layers and is_txt.shape[0] == b
    check(lib().cv_sparse_plan(ptr(is_txt), is_txt.stride(0), ptr(cur_len_dev), int(num_layers), b, int(window),
                               int(num_pivot), int(max_sequence_length), ptr(seed_dev), ptr(idx), nmax, ptr(n_dev),
                               ptr(err), stream_ptr()), "cv_sparse_plan")


def attn_decode_gather(qkv, cache, heads, cur_len_dev, idx, n_dev, *, nsplit=1, out=None, workspace=None):
    """attn_decode over the key list idx [b, nmax] int32 (first *n_dev entries; it contains the new token's position)."""
    require_cuda(qkv, cache, idx, n_dev, cur_len_dev)
    b, h3 = qkv.shape
    h = h3 // 3
    assert qkv.is_contiguous() and cache.stride(2) == 1 and cache.stride(1) == 2 * h and cache.shape[2] == 2 * h
    assert idx.dtype == torch.int32 and idx.shape[0] == b and idx.stride(1) == 1
    if out is None:
        out = torch.empty((b, h), dtype=torch.bfloat16, device=qkv.device)
    if nsplit > 1 and workspace is None:
        workspace = torch.empty(lib().cv_attn_decode_workspace_bytes(b, heads, nsplit) // 4, dtype=torch.float32,
                                device=qkv.device)
    rc = lib().cv_attn_decode_gather(ptr(qkv), ptr(cache), cache.stride(0), ptr(cur_len_dev), ptr(idx), idx.stride(0),
                                     ptr(n_dev), ptr(out), ptr(workspace), b, heads, 64, cache.shape[1], nsplit,
                                     stream_ptr())
    check(rc, "cv_attn_decode_gather")
    return out


def ln_pair_small_m(res_in, gemm_out, absmax_gemm, post, pre, eps, *, want_res_out=True):
    """y = res_in + LN_post(gemm_out) (gemm_out may be None), xn = LN_pre(y).  post/pre: (gamma, beta) bf16.
    Returns (y fp32 or None, xn bf16)."""
    require_cuda(res_in, gemm_out)
    M, K = res_in.shape
    assert res_in.dtype == torch.float32 and res_in.is_contiguous()
    y = torch.empty_like(res_in) if want_res_out else None
    xn = torch.empty((M, K), dtype=torch.bfloat16, device=res_in.device)
    gp, bp = post if post is not None else (None, None)
    rc = lib().cv_ln_pair_small_m(ptr(res_in), ptr(gemm_out), ptr(absmax_gemm), ptr(gp), ptr(bp), ptr(pre[0]),
                                  ptr(pre[1]), float(eps), ptr(y), ptr(xn), M, K, stream_ptr())
    check(rc, "cv_ln_pair_small_m")
    return y, xn


DECODE_STEP_MAX_BATCH = 8


def decode_step_workspace(hidden, heads, device):
    """Zeroed workspace of the persistent decode step (counters + L2-resident activations)."""
    n = lib().cv_decode_step_workspace_bytes(int(hidden), int(heads))
    if n <= 0:
        raise _lib.CogViewB200Error("cv_decode_step_workspace_bytes(%d, %d) failed" % (hidden, heads))
    return torch.zeros(n, dtype=torch.uint8, device=device)


def decode_step(layer_table, num_layers, heads, eps, eps_final, wte, wpe, lnf_g, lnf_b, ids, pos, cur_len, cache,
                logits, workspace, prof=None):
    """One token per sequence through every layer + logits in ONE kernel (cv_decode_step).
    layer_table: int64 [num_layers, 16] device tensor of parameter pointers in cv_decode_layer order;
    cache: [L, b, max_len, 2h] bf16; ids/pos: int64 [b(,1)]; cur_len: int32 [1]; logits: fp32 [b, V] (written)."""
    require_cuda(layer_table, wte, wpe, lnf_g, lnf_b, ids, pos, cur_len, cache, logits, workspace)
    L, b, max_len, h2 = cache.shape
    assert L == num_layers and cache.dtype == torch.bfloat16 and cache.stride(3) == 1 and cache.stride(2) == h2
    assert layer_table.dtype == torch.int64 and layer_table.shape == (num_layers, 16) and layer_table.is_contiguous()
    assert ids.dtype == torch.int64 and pos.dtype == torch.int64 and ids.numel() == b and pos.numel() == b
    assert ids.is_contiguous() and pos.is_contiguous() and cur_len.dtype == torch.int32
    assert logits.dtype == torch.float32 and logits.shape[0] == b and logits.stride(1) == 1
    assert wte.dtype == torch.bfloat16 and wte.is_contiguous() and wpe.is_contiguous()
    a = _lib.DecodeStepArgs(
        layers=ptr(layer_table), num_layers=num_layers, hidden=h2 // 2, heads=heads, vocab=wte.shape[0], batch=b,
        max_len=max_len, eps=float(eps), eps_final=float(eps_final), wte=ptr(wte), wpe=ptr(wpe), lnf_g=ptr(lnf_g),
        lnf_b=ptr(lnf_b), ids=ptr(ids), pos=ptr(pos), cur_len=ptr(cur_len), cache=ptr(cache),
        cache_layer_stride=cache.stride(0), cache_batch_stride=cache.stride(1), logits=ptr(logits),
        ld_logits=logits.stride(0), workspace=ptr(workspace), prof=ptr(prof))
    import ctypes
    check(lib().cv_decode_step(ctypes.byref(a), stream_ptr()), "cv_decode_step")
    return logits


def valid_ranges(invalid, vocab):
    """Complement of a list of [lo, hi) index pairs inside [0, vocab) as a sorted list of [lo, hi) pairs."""
    inv = sorted((max(0, int(a)), min(vocab, int(z))) for a, z in invalid)
    out, cur = [], 0
    for a, z in inv:
        if a > cur:
            out.append((cur, a))
        cur = max(cur, z)
    if cur < vocab:
        out.append((cur, vocab))
    return out


def sample_topk(logits, temperature, top_k, valid, *, seed=0, seed_dev=None, step=None, next_ids=None, out_tokens=None,
                score_acc=None, pos=None, cur_len=None, done=None, want_probs=False):
    """Sampling tail of generation/sampling.py:157-183 in one kernel.  logits fp32 [b, V] (unchanged);
    valid: list of [lo, hi) vocabulary ranges (<= 4).  Returns (next_ids int64 [b], probs or None)."""
    import ctypes
    require_cuda(logits, seed_dev, step, next_ids, out_tokens, score_acc, pos, cur_len, done)
    b, V = logits.shape
    assert logits.dtype == torch.float32 and logits.stride(1) == 1
    if not 1 <= len(valid) <= 4:
        raise _lib.CogViewB200Error("cv_sample_topk takes 1..4 valid vocabulary ranges, got %r" % (valid,))
    if next_ids is None:
        next_ids = torch.empty(b, dtype=torch.int64, device=logits.device)
    if (step is not None or cur_len is not None) and done is None:
        done = torch.zeros(1, dtype=torch.int32, device=logits.device)
    probs = torch.empty((b, logits.stride(0)), dtype=torch.float32, device=logits.device) if want_probs else None
    flat = (ctypes.c_int * (2 * len(valid)))(*[int(x) for r in valid for x in r])
    rc = lib().cv_sample_topk(ptr(logits), logits.stride(0), b, V, float(temperature), int(top_k), flat, len(valid),
                              int(seed) & 0xFFFFFFFFFFFFFFFF, ptr(seed_dev), ptr(step), ptr(next_ids), ptr(out_tokens),
                              0 if out_tokens is None else out_tokens.stride(0), ptr(score_acc), ptr(pos), ptr(cur_len),
                              ptr(done), ptr(probs), stream_ptr())
    check(rc, "cv_sample_topk")
    return next_ids, (probs[:, :V] if want_probs else None)


# ----------------------------------------------------------------------------------------------------
# VQ-VAE kernels (NHWC bf16 activations)
# ----------------------------------------------------------------------------------------------------
def conv2d_k4s2(x, w_packed, bias, relu):
    """x: [B, H, W, Cin] bf16 NHWC; w_packed: [16, Cout, Cin] bf16 -> [B, H/2, W/2, Cout] bf16."""
    require_cuda(x, w_packed, bias)
    B, H, W, Cin = x.shape
    Cout = w_packed.shape[1]
    assert x.is_contiguous() and w_packed.is_contiguous() and x.dtype == torch.bfloat16
    y = torch.empty((B, H // 2, W // 2, Cout), dtype=torch.bfloat16, device=x.device)
    check(lib().cv_conv2d_k4s2(ptr(x), ptr(w_packed), ptr(bias), ptr(y), B, H, W, Cin, Cout, int(relu), stream_ptr()),
          "cv_conv2d_k4s2")
    return y


def conv_transpose2d_k4s2(x, w_packed, bias, relu):
    """x: [B, H, W, Cin] bf16 NHWC; w_packed: [16, Cout, Cin] bf16 -> [B, 2H, 2W, Cout] bf16."""
    require_cuda(x, w_packed, bias)
    B, H, W, Cin = x.shape
    Cout = w_packed.shape[1]
    assert x.is_contiguous() and w_packed.is_contiguous() and x.dtype == torch.bfloat16
    y = torch.empty((B, 2 * H, 2 * W, Cout), dtype=torch.bfloat16, device=x.device)
    check(lib().cv_conv_transpose2d_k4s2(ptr(x), ptr(w_packed), ptr(bias), ptr(y), B, H, W, Cin, Cout, int(relu),
                                         stream_ptr()), "cv_conv_transpose2d_k4s2")
    return y


def im2col_k4s2_c3(img):
    """img: [B, 3, H, W] fp32 NCHW -> [B*(H/2)*(W/2), 64] bf16 patches (48 used)."""
    require_cuda(img)
    B, C, H, W = img.shape
    assert C == 3 and img.dtype == torch.float32 and img.is_contiguous()
    out = torch.empty((B * (H // 2) * (W // 2), 64), dtype=torch.bfloat16, device=img.device)
    check(lib().cv_im2col_k4s2_c3(ptr(img), ptr(out), B, H, W, stream_ptr()), "cv_im2col_k4s2_c3")
    return out


def vq_split3(z):
    require_cuda(z)
    rows, dim = z.shape
    assert z.dtype == torch.float32 and z.is_contiguous()
    out = torch.empty((rows, 3 * dim), dtype=torch.bfloat16, device=z.device)
    check(lib().cv_vq_split3(ptr(z), ptr(out), rows, dim, stream_ptr()), "cv_vq_split3")
    return out


def vq_argmin(scores, e2, z, codebook, margin=1e-4):
    require_cuda(scores, e2, z, codebook)
    rows, n_embed = scores.shape
    assert scores.dtype == torch.float32 and scores.stride(1) == 1 and codebook.is_contiguous() and z.is_contiguous()
    idx = torch.empty(rows, dtype=torch.int64, device=scores.device)
    check(lib().cv_vq_argmin(ptr(scores), scores.stride(0), ptr(e2), ptr(z), ptr(codebook), ptr(idx), rows, n_embed,
                             codebook.shape[1], float(margin), stream_ptr()), "cv_vq_argmin")
    return idx


def vq_lookup(idx, codebook, want_bf16=True, want_f32=False):
    require_cuda(idx, codebook)
    idx = idx.contiguous().view(-1)
    rows, dim = idx.numel(), codebook.shape[1]
    ob = torch.empty((rows, dim), dtype=torch.bfloat16, device=idx.device) if want_bf16 else None
    of = torch.empty((rows, dim), dtype=torch.float32, device=idx.device) if want_f32 else None
    check(lib().cv_vq_lookup(ptr(idx), ptr(codebook), ptr(ob), ptr(of), rows, dim, stream_ptr()), "cv_vq_lookup")
    return ob, of


def conv1x1_out3(x, w, bias, scale, shift):
    """x: [B, H, W, Cin] bf16 NHWC; w: [3, Cin] fp32 -> [B, 3, H, W] fp32 = (x.w + bias) * scale + shift."""
    require_cuda(x, w, bias, scale, shift)
    B, H, W, Cin = x.shape
    assert x.is_contiguous() and w.is_contiguous() and w.dtype == torch.float32
    out = torch.empty((B, 3, H, W), dtype=torch.float32, device=x.device)
    check(lib().cv_conv1x1_out3(ptr(x), ptr(w), ptr(bias), ptr(scale), ptr(shift), ptr(out), B, H, W, Cin,
                                stream_ptr()), "cv_conv1x1_out3")
    return out


def attn_gather(q, cache, idx, heads):
    """sparse_attention_inference: q [b, sq, h] view, cache [b, max_len, 2h] (K|V), idx [b, n] int64 -> [b, sq, h]."""
    require_cuda(q, cache, idx)
    b, sq, h = q.shape
    assert q.stride(2) == 1 and cache.stride(2) == 1 and cache.stride(1) == 2 * h and idx.dtype == torch.int64
    idx = idx.contiguous()
    out = torch.empty((b, sq, h), dtype=torch.bfloat16, device=q.device)
    rc = lib().cv_attn_gather(ptr(q), q.stride(1), q.stride(0), ptr(cache), cache.stride(0), ptr(idx), ptr(out), b, heads,
                              64, sq, idx.shape[1], stream_ptr())
    check(rc, "cv_attn_gather")
    return out
