"""Oracle vs the committed golden fixtures (generated from the live reference).  CPU only."""
import pytest
import torch

from oracle import rvsa_oracle as O
from tests.helpers import check_grads_against_golden, check_maps, load_golden


@pytest.mark.parametrize("name", ["tiny160", "tiny224"])
def test_oracle_forward_matches_golden(name):
    g = load_golden(name)
    with torch.no_grad():
        outs = O.backbone_forward(g["sd"], g["cfg"], g["x"])
    check_maps(outs, g["z"], "fwd", 2e-5)                # fp32 reassociation only


@pytest.mark.parametrize("name", ["tiny160", "tiny224"])
def test_oracle_backward_matches_golden(name):
    g = load_golden(name)
    P = {k: (v.clone().requires_grad_(True) if v.is_floating_point() else v) for k, v in g["sd"].items()}
    loss = O.synthetic_loss(O.backbone_forward(P, g["cfg"], g["x"]))
    assert abs(loss.item() - g["loss"]) < 1e-5
    loss.backward()
    grads = {k: v.grad for k, v in P.items() if v.is_floating_point()}
    check_grads_against_golden(grads, g, tol=2e-4)


def test_oracle_fp64_close_to_fp32():
    g = load_golden("tiny160")
    P64 = {k: (v.double() if v.is_floating_point() else v) for k, v in g["sd"].items()}
    with torch.no_grad():
        o64 = O.backbone_forward(P64, g["cfg"], g["x"].double())
    check_maps([o.float() for o in o64], g["z"], "fwd", 2e-5)


def test_zero_sampling_params_is_plain_window_attention():
    """SURVEY A.1 identity: off = scale = angle = 0 puts every tap on a pixel centre."""
    g = load_golden("tiny224")
    P = dict(g["sd"])
    pre = "blocks.0.attn."
    for k in list(P):
        if k.startswith(pre + "sampling_"):
            P[k] = torch.zeros_like(P[k])
    torch.manual_seed(0)
    xn = torch.randn(2, 196, 128)
    got = O.rvsa_attention(xn, P, pre, 14, 14, 2)
    # plain 7x7 window attention with the same rel-pos terms
    B, N, C, nH, hd = 2, 196, 128, 2, 64
    qkv = (xn @ P[pre + "qkv.weight"].t() + P[pre + "qkv.bias"]).reshape(B, 2, 7, 2, 7, 3, nH, hd)
    qkv = qkv.permute(5, 0, 1, 3, 6, 2, 4, 7).reshape(3, B, 2, 2, nH, 49, hd)
    q, k, v = qkv[0], qkv[1], qkv[2]
    S = (q @ k.transpose(-1, -2)) * hd ** -0.5
    iy = torch.arange(7).repeat_interleave(7)
    ix = torch.arange(7).repeat(7)
    Rh = P[pre + "rel_pos_h"][iy[:, None] - iy[None, :] + 6]
    Rw = P[pre + "rel_pos_w"][ix[:, None] - ix[None, :] + 6]
    S = S + torch.einsum("...qc,qkc->...qk", q, Rh) + torch.einsum("...qc,qkc->...qk", q, Rw)
    idx = (iy[:, None] - iy[None, :] + 6) * 13 + (ix[:, None] - ix[None, :] + 6)
    S = S + P[pre + "relative_position_bias_table"][idx].permute(2, 0, 1)
    o = torch.softmax(S, -1) @ v                                              # (B,2,2,nH,49,hd)
    o = o.reshape(B, 2, 2, nH, 7, 7, hd).permute(0, 1, 4, 2, 5, 3, 6).reshape(B, N, C)
    want = o @ P[pre + "proj.weight"].t() + P[pre + "proj.bias"]
    assert float((got - want).abs().max()) < 1e-5


def test_flop_model_matches_survey():
    f = O.algorithmic_gflop_per_image(O.vit_l_config(224))
    assert abs(f["total"] - 130.20) < 0.05 and abs(f["attn_mlp"] - 119.95) < 0.05
    f = O.algorithmic_gflop_per_image(O.vit_b_config(224))
    assert abs(f["total"] - 39.87) < 0.05 and abs(f["attn_mlp"] - 34.07) < 0.05
