"""Drop-in boundary (CPU): constructor kwargs, state_dict layout, factories, registry, config files, init_weights.  What the reference
module and its fine-tuning configs showed is stored in tests/golden/reference_boundary.json (tests/golden/make_golden.py)."""
import json
import os
import types

import pytest
import torch

import mtp_b200
from mtp_b200 import checkpoint
from tests.helpers import GOLDEN_DIR, hashed_state_dict, tensor_sha256

with open(os.path.join(GOLDEN_DIR, "reference_boundary.json")) as _f:
    REF = json.load(_f)


def _tiny(**kw):
    base = dict(img_size=160, patch_size=16, embed_dim=128, depth=4, num_heads=2, mlp_ratio=4, qkv_bias=True,
                use_abs_pos_emb=True, interval=2, out_indices=[0, 1, 2, 3], drop_path_rate=0.1, use_rel_pos_bias=True)
    base.update(kw)
    return base


def test_factories_and_param_budget():
    """[V]:819-865: ViT-B 93.29 M params / 245 state_dict entries; ViT-L 317,628,800 params in 489 tensors (SURVEY B.3)."""
    with torch.device("meta"):
        b = mtp_b200.vit_b_rvsa(types.SimpleNamespace(image_size=224, use_ckpt="False"))
        l = mtp_b200.vit_l_rvsa(types.SimpleNamespace(image_size=224, use_ckpt="True"))
    assert sum(p.numel() for p in b.parameters()) == 93291328 and len(b.state_dict()) == 245
    assert sum(p.numel() for p in l.parameters()) == 317628800 and len(list(l.parameters())) == 489
    assert l.use_checkpoint and not b.use_checkpoint
    assert b.out_channels == [768] * 4 and l.out_channels == [1024] * 4
    assert b.get_num_layers() == 12 and b.no_weight_decay() == {"pos_embed", "cls_token"}
    assert b.patch_embed.patch_shape == (14, 14)
    assert [blk.window for blk in b.blocks] == [(i + 1) % 3 != 0 for i in range(12)]
    assert abs(l.blocks[-1].drop_path_prob - 0.1) < 1e-7 and l.blocks[0].drop_path_prob == 0.0


def test_layer_decay_names_are_parseable():
    """mmcv_custom/layer_decay_optimizer_constructor_vit.py:7-16 parses backbone.blocks.<i>. / patch_embed / pos_embed."""
    from mtp_b200.trainer import layer_decay_group
    with torch.device("meta"):
        m = mtp_b200.ViT_Win_RVSA_V3_WSZ7(**_tiny())
    ids = {n: layer_decay_group(n, tuple(p.shape), 6, "backbone.") for n, p in m.named_parameters()}
    assert ids["pos_embed"] == (0, True) and ids["patch_embed.proj.weight"] == (0, False)
    assert ids["blocks.2.attn.qkv.weight"] == (3, False) and ids["blocks.2.norm1.weight"] == (3, True)
    assert ids["fpn1.0.weight"][0] == 5
    # pretrain quirk: names start with "encoder." so everything lands in the last layer
    assert all(layer_decay_group(n, tuple(p.shape), 6, "encoder.")[0] == 5 for n, p in m.named_parameters())


@pytest.mark.parametrize("img", [160, 224])
def test_state_dict_round_trip_with_reference(img):
    ref = REF["state_dict_layout"][str(img)]
    new = mtp_b200.ViT_Win_RVSA_V3_WSZ7(**_tiny(img_size=img))
    ns = new.state_dict()
    assert [k for k, _, _ in ref["keys"]] == list(ns.keys())
    for k, shape, dtype in ref["keys"]:
        assert list(ns[k].shape) == shape and str(ns[k].dtype) == dtype, k
    assert tensor_sha256(ns["blocks.0.attn.relative_position_index"]) == ref["relative_position_index_sha256"]
    rs = {k: torch.zeros(shape, dtype=getattr(torch, dtype[len("torch."):])) for k, shape, dtype in ref["keys"]}
    new.load_state_dict(rs, strict=True)                    # a state_dict of the reference's layout loads strictly
    assert [n for n, _ in new.named_parameters()] == ref["parameters"]


def test_init_statistics_match_reference():
    """Same init recipe ([V]:676-691): trunc-normal(.02) linears, proj/fc2 rescaled by 1/sqrt(2*layer_id), LN = (1, 0)."""
    torch.manual_seed(0)
    n = mtp_b200.ViT_Win_RVSA_V3_WSZ7(**_tiny())
    for k, ref_std in REF["init_std"].items():
        assert abs(ref_std - n.state_dict()[k].std().item()) < 0.1 * ref_std, k
    assert float(n.blocks[1].norm1.weight.min()) == 1.0 and float(n.blocks[1].norm1.bias.abs().max()) == 0.0
    assert float(n.blocks[0].attn.rel_pos_h.abs().max()) == 0.0            # zero-initialised tables ([V]:216-217)


def test_every_finetune_config_builds():
    """Every RS_Tasks_Finetune/**/configs/mtp/**/*rvsa*.py backbone dict constructs the matching twin (meta device)."""
    ft = REF["finetune_configs"]
    assert len(ft["files"]) >= 60
    built = 0
    for entry in ft["backbones"]:
        cfg = dict(entry["backbone"])
        name = cfg.pop("type")
        cfg["type"] = f"{entry['toolkit']}.{name}"
        with torch.device("meta"):
            m = mtp_b200.MODELS.build(cfg)
        assert m.embed_dim in (768, 1024) and m.patch_embed.patch_shape[0] == cfg["img_size"] // 16
        built += 1
    assert built >= 60


def test_registry_flavours():
    with torch.device("meta"):
        seg = mtp_b200.MODELS.build(dict(type="RVSA_MTP", **_tiny()))
        det = mtp_b200.MODELS.build(dict(type="mmdet.RVSA_MTP", **_tiny(out_indices=[3])))
        br = mtp_b200.MODELS.build(dict(type="RVSA_MTP_branches", **_tiny()))
        cls = mtp_b200.MODELS.build(dict(type="mmpretrain.RVSA_MTP", **_tiny()))
    assert not hasattr(seg, "norm") and seg.return_tuple and seg.apply_fpn
    assert det.feature_mode == "last_norm" and not any("full_attn_rel_pos" in n for n, _ in det.named_parameters())
    assert br.feature_mode == "multi" and not br.full_attn_rel_pos
    assert not cls.apply_fpn and hasattr(cls, "norm")
    assert mtp_b200.register_all() == {}              # no OpenMMLab toolkit is installed in this image
    with pytest.raises(KeyError):
        mtp_b200.MODELS.build(dict(type="nope"))


def test_unsupported_options_fail_loudly():
    for bad in (dict(patch_size=8), dict(init_values=0.1), dict(drop_rate=0.1), dict(embed_dim=96, num_heads=2), dict(hybrid_backbone=object())):
        with pytest.raises((NotImplementedError, ValueError)):
            with torch.device("meta"):
                mtp_b200.ViT_Win_RVSA_V3_WSZ7(**_tiny(**bad))


def test_convert_state_dict_prefixes_and_resize():
    m = mtp_b200.RVSA_MTP(**_tiny(img_size=224))           # 14x14 grid, full-attn tables 27 x 64
    src = mtp_b200.ViT_Win_RVSA_V3_WSZ7(**_tiny(img_size=160))
    with torch.no_grad():
        for n, p in src.named_parameters():
            if "rel_pos" in n:
                p.normal_(0, 0.02)
    sd = {"module.encoder." + k: v for k, v in src.state_dict().items()}
    sd["module.encoder_extra.junk"] = torch.zeros(1)       # not under "encoder." -> dropped by the prefix filter ([V]:727-728)
    out = checkpoint.convert_state_dict(m, {"state_dict": sd}, variant="finetune")
    assert not any("junk" in k for k in out) and all(not k.startswith(("module.", "encoder.")) for k in out)
    assert out["pos_embed"].shape == (1, 196, 128)                  # no cls token in the checkpoint -> 0 extra tokens
    assert out["blocks.1.attn.full_attn_rel_pos_h"].shape == (27, 64)
    want = torch.nn.functional.interpolate(src.state_dict()["blocks.1.attn.full_attn_rel_pos_h"].reshape(1, 1, 19, 64), size=(27, 64),
                                           mode="bicubic", align_corners=False).squeeze()
    assert torch.equal(out["blocks.1.attn.full_attn_rel_pos_h"], want)
    msg = m.load_state_dict(out, strict=False)
    assert msg.missing_keys == [] and set(msg.unexpected_keys) == {"norm.weight", "norm.bias"}      # mmseg twin has no final norm
    # pretrain variant assumes one extra (cls) token, as MAE checkpoints have ([V]:749)
    pe = torch.randn(1, 1 + 100, 128)
    out2 = checkpoint.convert_state_dict(src, {"model": {"pos_embed": pe}}, variant="pretrain")
    assert torch.equal(out2["pos_embed"], pe[:, 1:])


def test_init_weights_matches_reference(tmp_path):
    """init_weights(path) on the new class == the reference's own init_weights on the same checkpoint ([V]:693-778)."""
    src = hashed_state_dict(mtp_b200.ViT_Win_RVSA_V3_WSZ7(**_tiny(img_size=160)).state_dict(), 3)
    # an MAE-style checkpoint: cls-token slot in pos_embed, no full-attention rel-pos tables (they are grid-size specific and
    # the pretrain-variant loader does not resize them: a size mismatch raises in the reference too)
    sd = {"encoder." + k: v for k, v in src.items() if "full_attn_rel_pos" not in k}
    sd["encoder.pos_embed"] = torch.cat([torch.zeros(1, 1, 128), src["pos_embed"]], 1)
    path = str(tmp_path / "ckpt.pth")
    torch.save({"state_dict": sd}, path)
    for img in (160, 224):                                 # same grid (strip cls token) and 10x10 -> 14x14 bicubic resize
        new = mtp_b200.ViT_Win_RVSA_V3_WSZ7(**_tiny(img_size=img))
        new.init_weights(path)
        ns = new.state_dict()
        for k, ref in REF["init_weights"][str(img)].items():
            assert list(ns[k].shape) == ref["shape"] and tensor_sha256(ns[k]) == ref["sha256"], (img, k)
