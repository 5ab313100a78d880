"""Pin the oracle against the reference module: the reference's results on hashed weights and inputs are stored in
tests/golden/reference_pinning.npz (tests/golden/make_golden.py, run against a checkout of the original project)."""
import os

import numpy as np
import pytest
import torch

import mtp_b200
from oracle import rvsa_oracle as O
from tests.helpers import GOLDEN_DIR, check_grads_against_golden, check_maps, hashed_state_dict, hashed_tensor


@pytest.fixture(scope="module")
def z():
    return np.load(os.path.join(GOLDEN_DIR, "reference_pinning.npz"))


def _kw(img, C, depth, nH, interval, oi, dpr=0.1):
    return dict(img_size=img, patch_size=16, embed_dim=C, depth=depth, num_heads=nH, mlp_ratio=4, qkv_bias=True,
                use_abs_pos_emb=True, interval=interval, out_indices=list(oi), drop_path_rate=dpr, use_rel_pos_bias=True)


def _weights(kw, seed):
    """The hashed weights the reference ran with (its state_dict layout equals the drop-in class's: tests/test_boundary_cpu.py)."""
    return hashed_state_dict(mtp_b200.ViT_Win_RVSA_V3_WSZ7(**kw).state_dict(), seed)


def test_config1_vit_b_224_forward(z):
    """BASELINE.json configs[0]: ViT-B backbone forward, 1x3x224x224 on CPU."""
    P = _weights(_kw(224, 768, 12, 12, 3, (3, 5, 7, 11)), seed=0)
    cfg = O.vit_b_config(224)
    with torch.no_grad():
        o = O.backbone_forward(P, cfg, hashed_tensor((1, 3, 224, 224), 0, "input"))
    check_maps(o, z, "vitb224", 1e-5)


@pytest.mark.parametrize("img", [160, 320, 512])        # pad cases Hp 10->14, 20->21, 32->35
def test_padded_grids(z, img):
    P = _weights(_kw(img, 128, 4, 2, 2, (0, 1, 2, 3)), seed=3)
    cfg = O.OracleConfig(img_size=img, embed_dim=128, depth=4, num_heads=2, interval=2, out_indices=(0, 1, 2, 3))
    with torch.no_grad():
        o = O.backbone_forward(P, cfg, hashed_tensor((2, 3, img, img), 0, "input"))
    check_maps(o, z, f"padded{img}", 2e-5)


def test_backward_all_params(z):
    sd = _weights(_kw(160, 128, 4, 2, 2, (0, 1, 2, 3)), seed=5)
    cfg = O.OracleConfig(img_size=160, embed_dim=128, depth=4, num_heads=2, interval=2, out_indices=(0, 1, 2, 3))
    P = {k: (v.clone().requires_grad_(True) if v.is_floating_point() else v) for k, v in sd.items()}
    loss = O.synthetic_loss(O.backbone_forward(P, cfg, hashed_tensor((2, 3, 160, 160), 0, "input")))
    assert abs(loss.item() - float(z["backward/loss"])) < 1e-5
    loss.backward()
    nograd = [str(k) for k in z["backward/nograd"]]
    assert all(k.startswith("norm.") for k in nograd)        # the reference's final norm never gets a gradient
    g = {"gnorm": {}, "gfull": {}, "gsamp": {}}
    for k in z.files:
        grp, _, name = k[len("backward/"):].partition("/")
        if k.startswith("backward/") and grp in g:
            g[grp][name] = float(z[k]) if grp == "gnorm" else torch.from_numpy(z[k])
    assert set(g["gnorm"]) | set(nograd) == {k for k, v in sd.items() if v.is_floating_point()}
    check_grads_against_golden({k: v.grad for k, v in P.items() if v.is_floating_point()}, g, tol=2e-4)


def test_drop_path_train_mode(z):
    """timm drop_path semantics: x * bernoulli(keep)/keep per sample, separate draws for attn and MLP branches."""
    kw = _kw(160, 128, 4, 2, 2, (0, 1, 2, 3), dpr=0.5)
    P = _weights(kw, seed=7)
    cfg = O.OracleConfig(img_size=160, embed_dim=128, depth=4, num_heads=2, interval=2, out_indices=(0, 1, 2, 3))
    keep = torch.from_numpy(z["droppath/keep"])          # (depth, 2, B): the multipliers the reference's drop_path applied
    with torch.no_grad():
        o = O.backbone_forward(P, cfg, hashed_tensor((4, 3, 160, 160), 0, "input"), keep=keep)
    check_maps(o, z, "droppath", 2e-5)
