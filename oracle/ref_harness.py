"""Import the UNMODIFIED reference — from /root/reference in the dev container, else from the verbatim copy
``oracle/make_ref.py`` ships to the GPU box under ``oracle/_ref/reference`` (git-ignored) — with the three oracle-side
shims of SURVEY.md §8c. TEST / BASELINE INFRASTRUCTURE ONLY: pins the oracle restatements, generates tests/golden/*, and
is what ``bench.py --impl reference`` times.

Shims (none alters arithmetic):
  A  flash_attn_func -> eager softmax attention in [B,S,H,D] layout (flash_attn has no CPU backend)
  B  DynamicCache.__getitem__ -> (keys, values) of a layer (transformers 5.x dropped tuple indexing)
  C  sdpa attention: slice a 4-D mask to the key length (the reference reuses the cond-sized all-ones mask)
"""
from __future__ import annotations

import os
import sys

import torch

_SHIPPED = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref", "reference")
REF = "/root/reference" if os.path.isdir("/root/reference/modeling") else _SHIPPED


def available() -> bool:
    return os.path.isdir(os.path.join(REF, "modeling"))


def _eager_flash(q, k, v, causal=False):
    assert not causal
    scale = q.shape[-1] ** -0.5
    qh, kh, vh = (t.transpose(1, 2) for t in (q, k, v))
    a = torch.softmax((qh * scale) @ kh.transpose(-1, -2), dim=-1)
    return (a @ vh).transpose(1, 2).contiguous()


def shim_transformers():
    """Shims B and C, once: what the reference's calls into transformers need (also for driving Qwen3 directly)."""
    from transformers import DynamicCache
    from transformers.modeling_utils import ALL_ATTENTION_FUNCTIONS

    if not hasattr(DynamicCache, "_bd_shim"):
        DynamicCache.__getitem__ = lambda s, i: (s.layers[i].keys, s.layers[i].values)
        DynamicCache._bd_shim = True
        _orig = ALL_ATTENTION_FUNCTIONS["sdpa"]

        def _sdpa(module, q, k, v, attention_mask=None, **kw):
            if attention_mask is not None and attention_mask.dim() == 4:
                attention_mask = attention_mask[..., : k.shape[-2]]
            return _orig(module, q, k, v, attention_mask=attention_mask, **kw)

        ALL_ATTENTION_FUNCTIONS["sdpa"] = _sdpa


_done = False
_ns = None


def import_reference():
    """Returns a namespace with the reference modules; applies the shims once. The reference's top-level package is
    called ``modeling`` — the same name as this repo's drop-in package — so it is imported with /root/reference first
    on sys.path and then moved out of ``sys.modules`` (the namespace keeps the module objects alive)."""
    global _done, _ns
    if not available():
        raise RuntimeError("reference not present (neither /root/reference nor oracle/_ref/reference: run oracle/make_ref.py "
                           "in the dev container)")
    if _ns is not None:
        return _ns
    import types

    # resolve transformers' lazy imports (qwen3 -> torchvision -> torch.library.register_fake -> inspect.getmodule) NOW:
    # inspect.getmodule walks sys.modules and chokes on a namespace package without __file__, which is what the reference's
    # top-level ``modeling`` is while it is being imported
    from transformers import AutoTokenizer, Qwen3Config, Qwen3ForCausalLM, set_seed  # noqa: F401
    from transformers.activations import ACT2FN  # noqa: F401
    try:
        import flash_attn  # noqa: F401
    except Exception:
        import importlib.machinery
        m = types.ModuleType("flash_attn")
        m.__spec__ = importlib.machinery.ModuleSpec("flash_attn", None)  # transformers probes find_spec("flash_attn")
        m.flash_attn_func = _eager_flash
        sys.modules["flash_attn"] = m
    mine = {k: v for k, v in sys.modules.items() if k == "modeling" or k.startswith("modeling.")}
    for k in mine:
        del sys.modules[k]
    # this repo's ``modeling`` is a regular package and would win over the reference's namespace package no matter
    # the sys.path order: hide the repo root (and cwd) while importing the reference
    repo_root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hidden = [(i, p) for i, p in enumerate(sys.path) if os.path.abspath(p or os.getcwd()) == repo_root]
    for _, p in hidden:
        sys.path.remove(p)
    sys.path.insert(0, REF)
    try:
        import modeling.vision_head.flow_head_parallel_x as fh
        import modeling.vision_head.sampling_x as sx
        import modeling.vision_encoder.autoencoder as ae
        import modeling.utils as mu
        import modeling.t2i_pipeline as t2i
    finally:
        sys.path.remove(REF)
        for i, p in hidden:
            sys.path.insert(min(i, len(sys.path)), p)
        for k in [k for k in sys.modules if k == "modeling" or k.startswith("modeling.")]:
            del sys.modules[k]
        sys.modules.update(mine)
    if REF not in sys.path:
        sys.path.append(REF)  # the reference's own `utils.fs` etc. stay importable, behind this repo's packages

    # shim A, per call: CPU tensors (flash_attn has no CPU backend) -> eager softmax attention; CUDA tensors keep the real
    # flash_attn kernel (a GPU box runs BOTH reference arms in one process: GPU-eager and the host-core baseline)
    _real_flash = getattr(fh, "flash_attn_func", None)

    def _flash(q, k, v, *a, **kw):
        if q.is_cuda and _real_flash is not None and _real_flash is not _eager_flash:
            return _real_flash(q, k, v, *a, **kw)
        return _eager_flash(q, k, v, causal=bool(kw.get("causal", a[2] if len(a) > 2 else False)))

    fh.flash_attn_func = _flash
    shim_transformers()
    _done = True
    _ns = types.SimpleNamespace(fh=fh, sx=sx, ae=ae, mu=mu, t2i=t2i)
    return _ns


def import_reference_mllm():
    """The reference's ``modeling/mllm.py`` (dev container only: it imports the reference's ``data`` package, which is not
    shipped to the GPU box). Used by tests/test_interleaved_cpu.py to pin the interleaved plan bookkeeping against the
    reference's own ``forward_inference_block_causal`` and to show that its text branch raises."""
    import_reference()
    mine = {k: v for k, v in sys.modules.items() if k == "modeling" or k.startswith("modeling.")}
    for k in mine:
        del sys.modules[k]
    repo_root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hidden = [(i, p) for i, p in enumerate(sys.path) if os.path.abspath(p or os.getcwd()) == repo_root]
    for _, p in hidden:
        sys.path.remove(p)
    sys.path.insert(0, REF)
    try:
        import modeling.mllm as mllm
    finally:
        sys.path.remove(REF)
        for i, p in hidden:
            sys.path.insert(min(i, len(sys.path)), p)
        for k in [k for k in sys.modules if k == "modeling" or k.startswith("modeling.")]:
            del sys.modules[k]
        sys.modules.update(mine)
    return mllm
