"""TEST INFRASTRUCTURE — imports the UNMODIFIED reference modules on CPU from oracle/_ref, where
oracle/build_ref.py (run by build()) places them.  Used by bench.py's reference arm (cpu_baseline.kind =
"reference") and by
oracle/make_golden.py to (a) validate the travelling restatement oracle/cogview_oracle.py against the
real reference and (b) generate the golden fixtures under tests/golden/.

Harness-side shims (no edits to the reference; SURVEY.md §8c):
  1. fake `apex`:  FusedLayerNorm = torch.nn.LayerNorm, FusedAdam = torch.optim.AdamW
     (imports at mpu/sparse_transformer.py:23, mpu/layers.py:28)
  2. fake `deepspeed` with checkpointing.is_configured() -> False (mpu/sparse_transformer.py:30,107,465)
  3. sys.modules['torch._six'] with `inf` (mpu/grads.py:22; removed in torch >= 2)
  4. on CPU, mpu.sparse_transformer.get_cuda_rng_tracker -> no-op fork(), because standard_attention
     forks the CUDA RNG unconditionally (mpu/sparse_transformer.py:667-669)
plus torch.distributed gloo world_size=1 and mpu.initialize_model_parallel(1).
"""
import contextlib
import os
import sys
import types

import torch

REFERENCE_ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")

_loaded = {}


def available():
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "mpu"))


def _install_shims():
    apex = types.ModuleType("apex")
    norm = types.ModuleType("apex.normalization")
    fln = types.ModuleType("apex.normalization.fused_layer_norm")
    fln.FusedLayerNorm = torch.nn.LayerNorm
    norm.fused_layer_norm = fln
    apex.normalization = norm
    opt = types.ModuleType("apex.optimizers")
    opt.FusedAdam = torch.optim.AdamW
    apex.optimizers = opt
    sys.modules.setdefault("apex", apex)
    sys.modules.setdefault("apex.normalization", norm)
    sys.modules.setdefault("apex.normalization.fused_layer_norm", fln)
    sys.modules.setdefault("apex.optimizers", opt)

    ds = types.ModuleType("deepspeed")
    ck = types.ModuleType("deepspeed.checkpointing")
    ck.is_configured = lambda: False
    ds.checkpointing = ck
    ds.add_config_arguments = lambda parser: parser
    sys.modules.setdefault("deepspeed", ds)
    sys.modules.setdefault("deepspeed.checkpointing", ck)

    six = types.ModuleType("torch._six")
    six.inf = float("inf")
    sys.modules.setdefault("torch._six", six)


class _NoRng:
    @contextlib.contextmanager
    def fork(self, *a, **k):
        yield


def load():
    """Returns a dict with the reference's `mpu`, `gpt2_modeling` (model) and `vqvae` modules."""
    if _loaded:
        return _loaded
    if not available():
        raise RuntimeError("reference tree not found at %s" % REFERENCE_ROOT)
    _install_shims()
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import torch.distributed as dist
    if not dist.is_initialized():
        # a private single-rank gloo group through a file store: independent of any torchrun rendezvous in the environment
        # (bench.py --impl reference is launched under torchrun for N > 1 and rank 0 alone does the work; with
        # TORCHELASTIC_USE_AGENT_STORE set, env:// and tcp:// would try to join the agent's store as a client and block)
        import tempfile
        store_file = os.path.join(tempfile.mkdtemp(prefix="cogview_ref_pg_"), "store")
        dist.init_process_group("gloo", init_method="file://" + store_file, rank=0, world_size=1)
    import mpu  # noqa: the reference's package
    import mpu.sparse_transformer as st
    mpu.initialize_model_parallel(1)
    if torch.cuda.is_available():
        # a CUDA box (the GPU host timing the CPU arm): do what the reference's own entry points do before building the
        # model (pretrain_gpt2.py set_random_seed -> mpu.model_parallel_cuda_manual_seed), so that the RNG tracker that
        # standard_attention forks (mpu/sparse_transformer.py:667-669) knows its 'model-parallel-rng' state
        mpu.model_parallel_cuda_manual_seed(1234)
    else:
        st.get_cuda_rng_tracker = lambda: _NoRng()
    from model import gpt2_modeling
    import vqvae.api as vq_api
    import vqvae.vqvae_zc as vq_zc
    _loaded.update(mpu=mpu, sparse_transformer=st, gpt2_modeling=gpt2_modeling, vq_api=vq_api, vq_zc=vq_zc)
    return _loaded


def unload_paths():
    """Remove the reference from sys.path / sys.modules so the repo's own `mpu`-mirror can be imported."""
    if REFERENCE_ROOT in sys.path:
        sys.path.remove(REFERENCE_ROOT)
