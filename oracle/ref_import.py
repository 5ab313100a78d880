"""Import the UNMODIFIED reference backbone module for oracle pinning.  TEST INFRASTRUCTURE ONLY.

Used by tests/golden/make_golden.py, which takes the root of a checkout of the original project (``--reference DIR``) and
stores what the tests compare against under tests/golden/; the tests themselves never import it.  The reference file needs three
``timm`` helpers and one ``mmengine`` helper that are not installed; tiny shims with the documented
semantics (timm 0.9.x ``drop_path``/``to_2tuple``/``trunc_normal_``; ``get_dist_info`` -> (0, 1)) are put
into ``sys.modules`` before ``importlib`` executes the file where it lies (SURVEY.md Appendix D).
Nothing from the reference is copied into this repository.
"""
import collections.abc
import importlib.util
import os
import sys
import types

import torch

REF_FILE = "Multi-Task_Pretrain/backbone/vit_win_rvsa_v3_wsz7.py"      # relative to the root of the original project


# When a test wants a deterministic train-mode comparison it fills this queue with per-call (B,) multipliers
# (already divided by keep); the shim then consumes them in call order (attn branch, then MLP branch, per block).
KEEP_QUEUE: list = []


def _drop_path(x, drop_prob: float = 0.0, training: bool = False, scale_by_keep: bool = True):
    if drop_prob == 0.0 or not training:
        return x
    if KEEP_QUEUE:
        return x * KEEP_QUEUE.pop(0).reshape((x.shape[0],) + (1,) * (x.ndim - 1)).to(x.dtype)
    keep = 1 - drop_prob
    r = x.new_empty((x.shape[0],) + (1,) * (x.ndim - 1)).bernoulli_(keep)
    if keep > 0 and scale_by_keep:
        r.div_(keep)
    return x * r


def load_reference_module(root):
    path = os.path.join(root, REF_FILE)
    if not os.path.isfile(path):
        raise FileNotFoundError(path)
    if "ref_rvsa" in sys.modules:
        return sys.modules["ref_rvsa"]
    tl = types.ModuleType("timm.models.layers")
    tl.to_2tuple = lambda x: tuple(x) if isinstance(x, collections.abc.Iterable) and not isinstance(x, str) else (x, x)
    tl.trunc_normal_ = lambda t, mean=0.0, std=1.0, a=-2.0, b=2.0: torch.nn.init.trunc_normal_(t, mean, std, a, b)
    tl.drop_path = _drop_path
    md = types.ModuleType("mmengine.dist")
    md.get_dist_info = lambda: (0, 1)
    for name, mod in (("timm", types.ModuleType("timm")), ("timm.models", types.ModuleType("timm.models")),
                      ("timm.models.layers", tl), ("mmengine", types.ModuleType("mmengine")), ("mmengine.dist", md)):
        sys.modules.setdefault(name, mod)
    spec = importlib.util.spec_from_file_location("ref_rvsa", path)
    ref = importlib.util.module_from_spec(spec)
    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()):
        spec.loader.exec_module(ref)
    sys.modules["ref_rvsa"] = ref
    return ref


def build_reference(root, cfg_kwargs: dict, seed: int = 0):
    """Instantiate the reference class with ``cfg_kwargs`` and re-draw the zero-initialised rel-pos tables
    (they are ``zeros`` at init, [V]:83-84,216-217, which would leave the rel-pos terms untested)."""
    import contextlib
    import io
    ref = load_reference_module(root)
    torch.manual_seed(seed)
    with contextlib.redirect_stdout(io.StringIO()):
        model = ref.ViT_Win_RVSA_V3_WSZ7(**cfg_kwargs)
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if "rel_pos" in name:
                p.copy_(torch.randn(p.shape, generator=g) * 0.02)
            elif "sampling_" in name:
                # default Conv2d init is already non-zero; enlarge so offsets/scales/angles move taps noticeably
                p.mul_(4.0)
            elif name.endswith(".bias") or "norm" in name or ".ln." in name:
                # biases / LN affine init to 0 / 1: perturb so they are exercised
                p.add_(torch.randn(p.shape, generator=g) * 0.02)
    return model.eval()
