"""Generate the golden fixtures from the LIVE reference module (the original project's code, unmodified).

    python tests/golden/make_golden.py --reference DIR [tiny] [pinning] [boundary]     # DIR: root of a checkout of the original project

tiny      ``tests/golden/<name>.npz`` for each tiny configuration: the unmodified reference class ([V], imported by
          oracle/ref_import.py) is built with a fixed seed, run forward (eval) and forward+backward on a fixed input, and the batch
          size, the L2 norm of every state_dict entry and of the input (tests/helpers.golden_inputs regenerates both; checked here
          bit for bit), the four output maps (shape, TINY_MAP_SAMPLES entries, channel means), the loss (oracle.synthetic_loss)
          and, per parameter, the gradient's L2 norm plus GRAD_SAMPLES evenly spaced entries (full tensors for parameters with
          <= FULL_GRAD_MAX elements) are written.
pinning   ``tests/golden/reference_pinning.npz``, what tests/test_oracle_vs_reference.py compares the oracle with: the reference run on
          hashed weights and inputs (tests/helpers.py regenerates them), keeping per output map its shape, MAP_SAMPLES entries and its
          channel means, and per parameter gradient the norm and samples.
boundary  ``tests/golden/reference_boundary.json``, what tests/test_boundary_cpu.py compares the drop-in class with: the reference's
          state_dict layout, init statistics, the init_weights() results on a hashed checkpoint and the backbone dicts of the
          fine-tuning configs.
"""
import argparse
import ast
import contextlib
import glob
import io
import json
import os
import re
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref_import  # noqa: E402
from oracle.rvsa_oracle import synthetic_loss  # noqa: E402
from tests.helpers import TINY_MAP_SAMPLES, golden_inputs, hashed_state_dict, hashed_tensor, map_summary, tensor_sha256  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
GRAD_SAMPLES = 256
FULL_GRAD_MAX = 4096
PIN_FULL_GRAD_MAX = 1024

CONFIGS = {
    # name: (img_size, embed_dim, depth, heads, interval, out_indices, batch)
    "tiny160": dict(img_size=160, embed_dim=128, depth=4, num_heads=2, interval=2, out_indices=[0, 1, 2, 3], batch=2),
    "tiny224": dict(img_size=224, embed_dim=128, depth=4, num_heads=2, interval=2, out_indices=[0, 1, 2, 3], batch=1),
}


def ref_kwargs(c):
    return dict(img_size=c["img_size"], patch_size=16, embed_dim=c["embed_dim"], depth=c["depth"],
                num_heads=c["num_heads"], mlp_ratio=4, qkv_bias=True, use_abs_pos_emb=True, interval=c["interval"],
                out_indices=list(c["out_indices"]), drop_path_rate=0.1, use_rel_pos_bias=True)


def sample_idx(n):
    return np.unique(np.linspace(0, n - 1, min(n, GRAD_SAMPLES)).astype(np.int64))


def grad_summary(model, full_max):
    """gnorm/<k>, and gfull/<k> (<= full_max elements) or gsamp/<k> (GRAD_SAMPLES entries) for every parameter with a gradient."""
    blob = {}
    for k, p in model.named_parameters():
        if p.grad is None:
            continue
        g = p.grad.reshape(-1).double().numpy()
        blob["gnorm/" + k] = np.float64(np.sqrt((g * g).sum()))
        if g.size <= full_max:
            blob["gfull/" + k] = p.grad.numpy()
        else:
            blob["gsamp/" + k] = g[sample_idx(g.size)].astype(np.float32)
    return blob


def tiny(root):
    for name, c in CONFIGS.items():
        model = ref_import.build_reference(root, ref_kwargs(c), seed=0)
        torch.manual_seed(1234)
        x = torch.randn(c["batch"], 3, c["img_size"], c["img_size"])
        sd, x2 = golden_inputs(name, c["batch"])
        assert torch.equal(x, x2) and sd.keys() == model.state_dict().keys()
        assert all(torch.equal(v, model.state_dict()[k]) for k, v in sd.items()), "golden_inputs no longer reproduces the reference's init"
        with torch.no_grad():
            outs = model(x)
        model.zero_grad()
        loss = synthetic_loss(model(x))
        loss.backward()
        blob = {"batch": np.int64(c["batch"]), "loss": np.float64(loss.item()), "norm/x": np.float64(x.double().norm())}
        blob.update({"norm/" + k: np.float64(v.double().norm()) for k, v in sd.items()})
        for i, o in enumerate(outs):
            for f, v in map_summary(o, TINY_MAP_SAMPLES).items():
                blob[f"fwd/out{i}/{f}"] = v
        blob.update(grad_summary(model, FULL_GRAD_MAX))
        path = os.path.join(HERE, name + ".npz")
        np.savez_compressed(path, **blob)
        print(name, "loss", loss.item(), "->", path, os.path.getsize(path) // 1024, "KiB")


# ---------------------------------------------------------------------------------------------- reference_pinning.npz
def pin_kwargs(img, C, depth, nH, interval, oi, dpr=0.1):
    return dict(img_size=img, patch_size=16, embed_dim=C, depth=depth, num_heads=nH, mlp_ratio=4, qkv_bias=True,
                use_abs_pos_emb=True, interval=interval, out_indices=list(oi), drop_path_rate=dpr, use_rel_pos_bias=True)


def hashed_reference(root, kw, seed):
    m = ref_import.build_reference(root, kw, seed=seed)
    m.load_state_dict(hashed_state_dict(m.state_dict(), seed), strict=True)
    return m


def pinning(root):
    blob = {}

    def put(prefix, outs):
        for i, o in enumerate(outs):
            for f, v in map_summary(o).items():
                blob[f"{prefix}/out{i}/{f}"] = v

    # BASELINE.json configs[0]: ViT-B backbone forward at 224^2
    m = hashed_reference(root, pin_kwargs(224, 768, 12, 12, 3, (3, 5, 7, 11)), seed=0)
    with torch.no_grad():
        put("vitb224", m(hashed_tensor((1, 3, 224, 224), 0, "input")))
    # padded grids: Hp 10->14, 20->21, 32->35
    for img in (160, 320, 512):
        m = hashed_reference(root, pin_kwargs(img, 128, 4, 2, 2, (0, 1, 2, 3)), seed=3)
        with torch.no_grad():
            put(f"padded{img}", m(hashed_tensor((2, 3, img, img), 0, "input")))
    # gradients of every parameter
    m = hashed_reference(root, pin_kwargs(160, 128, 4, 2, 2, (0, 1, 2, 3)), seed=5)
    loss = synthetic_loss(m(hashed_tensor((2, 3, 160, 160), 0, "input")))
    loss.backward()
    blob["backward/loss"] = np.float64(loss.item())
    blob["backward/nograd"] = np.array([k for k, p in m.named_parameters() if p.grad is None])
    blob.update({"backward/" + k: v for k, v in grad_summary(m, PIN_FULL_GRAD_MAX).items()})
    # DropPath in train mode, timm semantics, with fixed per-sample multipliers
    B = 4
    m = hashed_reference(root, pin_kwargs(160, 128, 4, 2, 2, (0, 1, 2, 3), dpr=0.5), seed=7).train()
    rates = [r.item() for r in torch.linspace(0, 0.5, 4)]
    g = torch.Generator().manual_seed(11)
    keep = torch.ones(4, 2, B)
    for i, r in enumerate(rates):
        if r > 0:
            keep[i] = torch.bernoulli(torch.full((2, B), 1 - r), generator=g) / (1 - r)
    # block 0 has drop_prob 0 -> nn.Identity, no shim call
    ref_import.KEEP_QUEUE[:] = [keep[i, j] for i in range(1, 4) for j in range(2)]
    with torch.no_grad():
        put("droppath", m(hashed_tensor((B, 3, 160, 160), 0, "input")))
    assert not ref_import.KEEP_QUEUE
    blob["droppath/keep"] = keep.numpy()
    path = os.path.join(HERE, "reference_pinning.npz")
    np.savez_compressed(path, **blob)
    print("reference_pinning ->", path, os.path.getsize(path) // 1024, "KiB")


# ---------------------------------------------------------------------------------------------- reference_boundary.json
def tiny_kwargs(**kw):
    base = dict(img_size=160, patch_size=16, embed_dim=128, depth=4, num_heads=2, mlp_ratio=4, qkv_bias=True,
                use_abs_pos_emb=True, interval=2, out_indices=[0, 1, 2, 3], drop_path_rate=0.1, use_rel_pos_bias=True)
    base.update(kw)
    return base


def backbone_dicts(path):
    """Every `backbone=dict(...)` of a config file, without importing mmengine."""
    tree = ast.parse(open(path).read())
    out = []
    for node in ast.walk(tree):
        if isinstance(node, ast.keyword) and node.arg == "backbone" and isinstance(node.value, ast.Call):
            try:
                out.append({kw.arg: ast.literal_eval(kw.value) for kw in node.value.keywords})
            except Exception:
                pass
    return out


INIT_WEIGHTS_KEYS = ("pos_embed", "blocks.0.attn.qkv.weight", "blocks.2.attn.rel_pos_h", "fpn1.0.weight",
                     "blocks.0.attn.sampling_offsets.2.weight")


def boundary(root):
    out = {"state_dict_layout": {}, "init_std": {}, "init_weights": {}}
    for img in (160, 224):
        sd = ref_import.build_reference(root, tiny_kwargs(img_size=img), seed=0).state_dict()
        ref = ref_import.build_reference(root, tiny_kwargs(img_size=img), seed=0)
        out["state_dict_layout"][str(img)] = {
            "keys": [[k, list(v.shape), str(v.dtype)] for k, v in sd.items()],
            "parameters": [n for n, _ in ref.named_parameters()],
            "relative_position_index_sha256": tensor_sha256(sd["blocks.0.attn.relative_position_index"])}
    # the reference's own initialisation ([V]:676-691)
    mod = ref_import.load_reference_module(root)
    torch.manual_seed(0)
    with contextlib.redirect_stdout(io.StringIO()):
        sd = mod.ViT_Win_RVSA_V3_WSZ7(**tiny_kwargs()).state_dict()
    for k in ("blocks.0.attn.qkv.weight", "blocks.3.attn.proj.weight", "blocks.3.mlp.fc2.weight", "pos_embed"):
        out["init_std"][k] = sd[k].std().item()
    # init_weights(path) on an MAE-style checkpoint: cls-token slot in pos_embed, no full-attention rel-pos tables
    src = hashed_state_dict(ref_import.build_reference(root, tiny_kwargs(img_size=160), seed=3).state_dict(), 3)
    ck = {"encoder." + k: v for k, v in src.items() if "full_attn_rel_pos" not in k}
    ck["encoder.pos_embed"] = torch.cat([torch.zeros(1, 1, 128), src["pos_embed"]], 1)
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "ckpt.pth")
        torch.save({"state_dict": ck}, path)
        for img in (160, 224):                              # same grid (strip cls token) and 10x10 -> 14x14 bicubic resize
            ref = ref_import.build_reference(root, tiny_kwargs(img_size=img), seed=9)
            with contextlib.redirect_stdout(io.StringIO()):
                ref.init_weights(path)
            rs = ref.state_dict()
            out["init_weights"][str(img)] = {k: {"shape": list(rs[k].shape), "sha256": tensor_sha256(rs[k])} for k in INIT_WEIGHTS_KEYS}
    # every RS_Tasks_Finetune/**/configs/mtp/**/*rvsa*.py backbone dict of an RVSA_MTP type
    ft = os.path.join(root, "RS_Tasks_Finetune")
    files = sorted(glob.glob(os.path.join(ft, "**", "configs", "mtp", "**", "*rvsa*.py"), recursive=True))
    cfgs = []
    for f in files:
        rel = os.path.relpath(f, ft)
        tk = ("mmseg" if "Semantic_Segmentation" in f else "mmpretrain" if "Scene_Classification" in f else
              "opencd" if "Change_Detection" in f else "mmdet" if "Horizontal_Detection" in f else "mmrotate")
        cfgs += [{"file": rel, "toolkit": tk, "backbone": c} for c in backbone_dicts(f) if str(c.get("type", "")).startswith("RVSA_MTP")]
    out["finetune_configs"] = {"files": [os.path.relpath(f, ft) for f in files], "backbones": cfgs}
    path = os.path.join(HERE, "reference_boundary.json")
    text = json.dumps(out, indent=1)
    text = re.sub(r"\[\s+([^\[\]{}\"]*?)\s+\]", lambda mt: "[" + re.sub(r"\s+", " ", mt.group(1)) + "]", text)     # number lists on one line
    text = re.sub(r"\[\s+(\"[^\"]*\"),\s+(\[[^\[\]]*\]),\s+(\"[^\"]*\")\s+\]", r"[\1, \2, \3]", text)           # [name, shape, dtype]
    with open(path, "w") as fh:
        fh.write(text + "\n")
    print("reference_boundary ->", path, os.path.getsize(path) // 1024, "KiB")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", required=True, help="root of a checkout of the original project")
    ap.add_argument("what", nargs="*", choices=["tiny", "pinning", "boundary"], default=["tiny", "pinning", "boundary"])
    a = ap.parse_args()
    for w in a.what:
        globals()[w](a.reference)


if __name__ == "__main__":
    main()
