"""CPU oracle for the ViT + RVSA backbone hot path.  TEST INFRASTRUCTURE ONLY.

This file is the parity checker: a plain fp32/fp64 PyTorch *functional* restatement of the
reference module ``Multi-Task_Pretrain/backbone/vit_win_rvsa_v3_wsz7.py`` (called ``[V]`` below),
written from the closed-form math in SURVEY.md Appendix A, not from the reference's op sequence.
Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline / ``--impl reference``
legs may import it.  The product path (``mtp_b200``) never does, and fails loudly when its CUDA
library is missing.

Pinning: the reference ships no tests or golden vectors for this path (SURVEY.md §4), so the oracle
is pinned against the *live* reference module, imported unmodified (``oracle/ref_import.py``) by
``tests/golden/make_golden.py``, which stores the reference's results under ``tests/golden/``;
``tests/test_oracle_vs_reference.py`` and ``tests/test_oracle_golden.py`` compare the oracle with them.

All functions take the reference's ``state_dict`` key layout ([V] module tree, SURVEY.md §8b).
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence

import torch
import torch.nn.functional as F

WS = 7  # window size is hard-wired to 7 in the reference ([V]:629 ``window_size=(7, 7)``)


@dataclass
class OracleConfig:
    """Mirror of the constructor arguments that change arithmetic ([V]:590-594)."""
    img_size: int = 224
    patch_size: int = 16
    in_chans: int = 3
    embed_dim: int = 768
    depth: int = 12
    num_heads: int = 12
    mlp_ratio: float = 4.0
    interval: int = 3
    out_indices: Sequence[int] = (3, 5, 7, 11)
    # finetune-variant switches (SURVEY.md §2.2)
    full_attn_rel_pos: bool = True      # mmdet/mmrotate twins disable it
    feature_mode: str = "multi"          # "multi" ([V]:804) | "last_norm" (mmdet RVSA_MTP)
    apply_fpn: bool = True               # mmpretrain / opencd twins skip the fpn ops
    ln_eps: float = 1e-6
    # Test aid, not part of the reference: round to bf16 (straight-through for autograd) at exactly the points where the
    # CUDA path stores bf16 (GEMM operands: weights, LN outputs, qkv, attention output, GELU output, fpn intermediates).
    # With it the oracle predicts the CUDA path's forward to ~1e-3 and shares its bilinear-tap cell decisions.
    emulate_bf16: bool = False
    # Test aid: additionally round the COTANGENTS to bf16 where the CUDA backward stores them as bf16 GEMM operands (branch
    # cotangents, dh, dy, dO, dS / P of the attention backward, dqkv, the pyramid intermediates) and differentiate GELU at the
    # bf16-rounded pre-activation the CUDA path keeps.  Makes the oracle's backward carry the same rounding-noise SOURCES as the CUDA
    # backward (it cannot reproduce the individual rounding decisions at depth: see tests/test_rounding_chaos_cpu.py).
    emulate_bf16_grad: bool = False

    @property
    def grid(self) -> int:
        return self.img_size // self.patch_size

    def is_window_block(self, i: int) -> bool:
        return (i + 1) % self.interval != 0          # [V]:629


def vit_b_config(img_size=224, **kw) -> OracleConfig:      # [V]:819-841
    return OracleConfig(img_size=img_size, embed_dim=768, depth=12, num_heads=12, interval=3,
                        out_indices=(3, 5, 7, 11), **kw)


def vit_l_config(img_size=224, **kw) -> OracleConfig:      # [V]:843-865
    return OracleConfig(img_size=img_size, embed_dim=1024, depth=24, num_heads=16, interval=6,
                        out_indices=(7, 11, 15, 23), **kw)


# ----------------------------------------------------------------------------------------------
# elementary pieces
# ----------------------------------------------------------------------------------------------

def _ste_bf16(t: torch.Tensor) -> torch.Tensor:
    """Round to bf16 in the forward pass, identity in the backward pass."""
    return t + (t.to(torch.bfloat16).to(t.dtype) - t).detach()


def _ident(t: torch.Tensor) -> torch.Tensor:
    return t


def _bf16(t: torch.Tensor) -> torch.Tensor:
    return t.to(torch.bfloat16).to(t.dtype)


class _RoundGrad(torch.autograd.Function):
    """Identity in the forward pass; rounds the cotangent to bf16 in the backward pass."""

    @staticmethod
    def forward(ctx, t):
        return t.view_as(t)

    @staticmethod
    def backward(ctx, g):
        return _bf16(g)


def _round_grad(t: torch.Tensor) -> torch.Tensor:
    return _RoundGrad.apply(t)


class _GeluSavedBf16(torch.autograd.Function):
    """erf-GELU of the fp32 pre-activation; the derivative is evaluated at the bf16 copy the CUDA path saves (fc1 epilogue out2)."""

    @staticmethod
    def forward(ctx, h):
        ctx.save_for_backward(_bf16(h))
        return gelu_erf(h)

    @staticmethod
    def backward(ctx, g):
        (hb,) = ctx.saved_tensors
        cdf = 0.5 * (1.0 + torch.erf(hb * (1.0 / math.sqrt(2.0))))
        pdf = torch.exp(-0.5 * hb * hb) * (1.0 / math.sqrt(2.0 * math.pi))
        return g * (cdf + hb * pdf)


class _AttnCoreBf16(torch.autograd.Function):
    """softmax(S) @ v with the bf16 staging of the tensor-core attention kernels, forward AND backward.
    ``normalized``: P is normalised before it is rounded (RVSA kernel) or rounded as exp(S - max) and O divided by the fp32 row sum
    (dense kernel).  Backward: dV = bf16(P)^T dO, dP = dO v^T, dS = bf16(P (dP - D))."""

    @staticmethod
    def forward(ctx, S, v, normalized):
        e = torch.exp(S - S.amax(-1, keepdim=True))
        ssum = e.sum(-1, keepdim=True)
        if normalized:
            O = _bf16(e / ssum) @ v
        else:
            O = (_bf16(e) @ v) / ssum
        ctx.save_for_backward(S, v, O)
        ctx.normalized = normalized
        return O

    @staticmethod
    def backward(ctx, dO):
        S, v, O = ctx.saved_tensors
        P = torch.softmax(S, dim=-1)
        dV = _bf16(P).transpose(-1, -2) @ dO
        dP = dO @ v.transpose(-1, -2)
        if ctx.normalized:
            D = (P * dP).sum(-1, keepdim=True)
        else:
            D = (dO * _bf16(O)).sum(-1, keepdim=True)
        return _bf16(P * (dP - D)), dV, None


def layer_norm(x: torch.Tensor, w: torch.Tensor, b: torch.Tensor, eps: float) -> torch.Tensor:
    """nn.LayerNorm(eps=1e-6) over the last dim ([V]:596)."""
    mu = x.mean(-1, keepdim=True)
    var = ((x - mu) ** 2).mean(-1, keepdim=True)
    return (x - mu) * torch.rsqrt(var + eps) * w + b


def gelu_erf(x: torch.Tensor) -> torch.Tensor:
    """nn.GELU() default = exact erf form ([V]:46,51)."""
    return 0.5 * x * (1.0 + torch.erf(x * (1.0 / math.sqrt(2.0))))


def patch_embed(x: torch.Tensor, w: torch.Tensor, b: torch.Tensor, p: int) -> torch.Tensor:
    """Conv2d(k=p, s=p) == per-patch GEMM ([V]:529,536-539).  Returns (B, N, C) tokens, row-major grid."""
    B, Cin, H, W = x.shape
    hp, wp = H // p, W // p
    x = x[:, :, :hp * p, :wp * p]
    patches = x.reshape(B, Cin, hp, p, wp, p).permute(0, 2, 4, 1, 3, 5).reshape(B, hp * wp, Cin * p * p)
    return patches @ w.reshape(w.shape[0], -1).t() + b


def window_padding(h: int, w: int):
    """Symmetric pad so (h+pad) % 7 == 0, extra pixel goes to bottom/right ([V]:298-303)."""
    pd_h = (WS - h % WS) % WS
    pd_w = (WS - w % WS) % WS
    pt, pl = pd_h // 2, pd_w // 2
    return pt, pd_h - pt, pl, pd_w - pl


def sampling_params(xn_grid: torch.Tensor, P: Dict[str, torch.Tensor], pre: str, nH: int, h: int, w: int):
    """Per-(image, window, head) offsets / scales / angle.  SURVEY.md A.1, [V]:228-243,347,354-368.

    xn_grid: (B, H', W', C) zero-padded normalised tokens.  Returns ox, oy, sx, sy, theta each (B, nh, nw, nH).
    """
    B, Hq, Wq, C = xn_grid.shape
    nh, nw = Hq // WS, Wq // WS
    pooled = xn_grid.reshape(B, nh, WS, nw, WS, C).mean(dim=(2, 4))          # zeros of the pad included
    a = torch.where(pooled >= 0, pooled, 0.01 * pooled)                        # LeakyReLU(0.01)
    def head(name, outc):
        wt = P[pre + f"{name}.2.weight"].reshape(outc, C)
        bs = P[pre + f"{name}.2.bias"]
        return a @ wt.t() + bs
    off = head("sampling_offsets", 2 * nH).reshape(B, nh, nw, nH, 2)
    sc = head("sampling_scales", 2 * nH).reshape(B, nh, nw, nH, 2)
    th = head("sampling_angles", nH)
    ox = off[..., 0] / (h // WS)            # sic: x divided by h//ws, y by w//ws ([V]:359-360)
    oy = off[..., 1] / (w // WS)
    return ox, oy, sc[..., 0], sc[..., 1], th


def bilinear_gather(m: torch.Tensor, px: torch.Tensor, py: torch.Tensor) -> torch.Tensor:
    """grid_sample(bilinear, zeros, align_corners=True) restated as a 4-tap gather ([V]:397-404).

    m: (G, Hq, Wq, D) value map; px, py: (G, S) pixel coords.  Returns (G, S, D).
    """
    G, Hq, Wq, D = m.shape
    x0 = torch.floor(px)
    y0 = torch.floor(py)
    fx = px - x0
    fy = py - y0
    flat = m.reshape(G, Hq * Wq, D)
    out = 0
    for dy, wy in ((0, 1 - fy), (1, fy)):
        for dx, wx in ((0, 1 - fx), (1, fx)):
            xi = x0 + dx
            yi = y0 + dy
            ok = (xi >= 0) & (xi <= Wq - 1) & (yi >= 0) & (yi <= Hq - 1)
            idx = (yi.clamp(0, Hq - 1) * Wq + xi.clamp(0, Wq - 1)).long()
            tap = torch.gather(flat, 1, idx.unsqueeze(-1).expand(G, idx.shape[1], D))
            out = out + tap * (wx * wy * ok.to(m.dtype)).unsqueeze(-1)
    return out


def rvsa_coords(ox, oy, sx, sy, th, Hq: int, Wq: int):
    """Sampling positions in pixels for every (image, head, padded-grid position).  SURVEY.md A.1.

    Inputs (B, nh, nw, nH).  Returns px, py of shape (B, nH, nh, 7, nw, 7).
    """
    dt, dev = ox.dtype, ox.device
    nh, nw = Hq // WS, Wq // WS
    lin_x = torch.linspace(-1, 1, Wq, dtype=dt, device=dev)
    lin_y = torch.linspace(-1, 1, Hq, dtype=dt, device=dev)
    refx = lin_x.reshape(nw, WS).mean(1)                                       # window centres [V]:317
    refy = lin_y.reshape(nh, WS).mean(1)
    k = torch.arange(WS, dtype=dt, device=dev)
    bx = k * 2 * WS / WS / (Wq - 1)
    bx = bx - bx.mean()                                                       # (i-3)*2/(W'-1)  [V]:326-329
    by = k * 2 * WS / WS / (Hq - 1)
    by = by - by.mean()

    def e(t):   # (B,nh,nw,nH) -> (B,nH,nh,1,nw,1)
        return t.permute(0, 3, 1, 2)[:, :, :, None, :, None]
    X = (1 + e(sx)) * bx[None, None, None, None, None, :]                      # [V]:372
    Y = (1 + e(sy)) * by[None, None, None, :, None, None]
    c, s = torch.cos(e(th)), torch.sin(e(th))
    cx = refx[None, None, None, None, :, None] + X * c - Y * s + e(ox)         # [V]:380-385
    cy = refy[None, None, :, None, None, None] + Y * c + X * s + e(oy)
    px = (cx + 1) * 0.5 * (Wq - 1)                                            # align_corners=True
    py = (cy + 1) * 0.5 * (Hq - 1)
    return px, py


def rvsa_attention(xn: torch.Tensor, P: Dict[str, torch.Tensor], pre: str, h: int, w: int, nH: int, r=_ident, gr=None) -> torch.Tensor:
    """RotatedVariedSizeWindowAttention.forward, [V]:287-433 / SURVEY.md A.1.  xn: LN'd (B, N, C).
    ``r`` is the identity (reference arithmetic) or the bf16 straight-through rounding of ``emulate_bf16``; ``gr`` (optional) rounds
    cotangents (``emulate_bf16_grad``)."""
    g_ = gr if gr is not None else _ident
    B, N, C = xn.shape
    hd = C // nH
    scale = hd ** -0.5
    pt, pb, pl, pr = window_padding(h, w)
    Hq, Wq = h + pt + pb, w + pl + pr
    nh, nw = Hq // WS, Wq // WS

    xg = F.pad(xn.reshape(B, h, w, C), (0, 0, pl, pr, pt, pb))                # zero pad  [V]:347
    ox, oy, sx, sy, th = sampling_params(xg, P, pre, nH, h, w)
    px, py = rvsa_coords(ox, oy, sx, sy, th, Hq, Wq)                           # (B,nH,nh,7,nw,7)

    # (the pooled sampling-head path above keeps an fp32 cotangent; the qkv GEMM's input cotangent dy1 is a bf16 tensor)
    qkv = g_(r(g_(xn) @ r(P[pre + "qkv.weight"]).t() + P[pre + "qkv.bias"]))         # [V]:390
    qkv = qkv.reshape(B, h, w, 3, nH, hd)
    qkv = F.pad(qkv, (0, 0, 0, 0, 0, 0, pl, pr, pt, pb))                        # zero pad AFTER bias [V]:392
    q, k, v = (qkv[:, :, :, i].permute(0, 3, 1, 2, 4) for i in range(3))        # (B,nH,Hq,Wq,hd)

    G = B * nH
    pxf = px.reshape(G, Hq * Wq)
    pyf = py.reshape(G, Hq * Wq)
    # (r: the tensor-core path stages the blended K~/V~ rows and the probabilities P as bf16 MMA operands)
    ks = r(bilinear_gather(k.reshape(G, Hq, Wq, hd), pxf, pyf)).reshape(B, nH, nh, WS, nw, WS, hd)
    vs = r(bilinear_gather(v.reshape(G, Hq, Wq, hd), pxf, pyf)).reshape(B, nH, nh, WS, nw, WS, hd)

    def win(t):  # (B,nH,nh,7,nw,7,hd) -> (B,nh,nw,nH,49,hd)
        return t.permute(0, 2, 4, 1, 3, 5, 6).reshape(B, nh, nw, nH, WS * WS, hd)
    qw = win(q.reshape(B, nH, nh, WS, nw, WS, hd))
    kw = win(ks)
    vw = win(vs)

    S = scale * (qw @ kw.transpose(-1, -2))                                     # [V]:410
    # decomposed rel-pos with the UNscaled q  ([V]:412 -> :176-191)
    iy = torch.arange(WS, device=xn.device).repeat_interleave(WS)               # token -> row in window
    ix = torch.arange(WS, device=xn.device).repeat(WS)
    Rh = P[pre + "rel_pos_h"][(iy[:, None] - torch.arange(WS, device=xn.device)[None, :]) + WS - 1]   # (49,7,hd)
    Rw = P[pre + "rel_pos_w"][(ix[:, None] - torch.arange(WS, device=xn.device)[None, :]) + WS - 1]
    rel_h = torch.einsum("...qc,qkc->...qk", qw, Rh)                            # (…,49,7) over key rows
    rel_w = torch.einsum("...qc,qkc->...qk", qw, Rw)
    S = S + rel_h[..., :, iy] + rel_w[..., :, ix]
    # learned bias table ([V]:414-418), index = (qy-jy+6)*13 + (qx-jx+6)  ([V]:272-282)
    idx = (iy[:, None] - iy[None, :] + WS - 1) * (2 * WS - 1) + (ix[:, None] - ix[None, :] + WS - 1)
    bias = P[pre + "relative_position_bias_table"][idx.reshape(-1)].reshape(WS * WS, WS * WS, nH).permute(2, 0, 1)
    S = S + bias
    if gr is not None:
        O = _AttnCoreBf16.apply(S, vw, True)
    else:
        A = r(torch.softmax(S, dim=-1))
        O = A @ vw                                                              # (B,nh,nw,nH,49,hd)
    O = O.reshape(B, nh, nw, nH, WS, WS, hd).permute(0, 1, 4, 2, 5, 3, 6).reshape(B, Hq, Wq, C)
    O = g_(r(O[:, pt:pt + h, pl:pl + w].reshape(B, N, C)))                      # crop  [V]:426
    return g_(O @ r(P[pre + "proj.weight"]).t() + P[pre + "proj.bias"])


def full_attention(xn: torch.Tensor, P: Dict[str, torch.Tensor], pre: str, h: int, w: int, nH: int,
                   use_rel_pos: bool = True, r=_ident, gr=None) -> torch.Tensor:
    """Attention.forward + calc_rel_pos_spatial, [V]:90-111,142-193 / SURVEY.md A.2."""
    g_ = gr if gr is not None else _ident
    B, N, C = xn.shape
    hd = C // nH
    scale = hd ** -0.5
    qkv = g_(r(g_(xn) @ r(P[pre + "qkv.weight"]).t() + P[pre + "qkv.bias"]))
    qkv = qkv.reshape(B, N, 3, nH, hd).permute(2, 0, 3, 1, 4)
    q, k, v = qkv[0] * scale, qkv[1], qkv[2]                                     # q scaled first [V]:100
    S = q @ k.transpose(-1, -2)
    if use_rel_pos:
        ty = torch.arange(h, device=xn.device).repeat_interleave(w)
        tx = torch.arange(w, device=xn.device).repeat(h)
        Rh = P[pre + "full_attn_rel_pos_h"][(ty[:, None] - torch.arange(h, device=xn.device)[None, :]) + h - 1]  # (N,h,hd)
        Rw = P[pre + "full_attn_rel_pos_w"][(tx[:, None] - torch.arange(w, device=xn.device)[None, :]) + w - 1]
        rel_h = torch.einsum("bnqc,qkc->bnqk", q, Rh)
        rel_w = torch.einsum("bnqc,qkc->bnqk", q, Rw)
        S = S + rel_h[..., :, ty] + rel_w[..., :, tx]
    if gr is not None:
        O = _AttnCoreBf16.apply(S, v, False)
    elif r is not _ident:
        # the dense tensor-core kernel stages exp(S - max) as a bf16 MMA operand and divides O by the fp32 row sum
        e = torch.exp(S - S.amax(-1, keepdim=True))
        O = (r(e) @ v) / e.sum(-1, keepdim=True)
    else:
        O = torch.softmax(S, dim=-1) @ v
    O = g_(r(O.transpose(1, 2).reshape(B, N, C)))
    return g_(O @ r(P[pre + "proj.weight"]).t() + P[pre + "proj.bias"])


def mlp(xn: torch.Tensor, P: Dict[str, torch.Tensor], pre: str, r=_ident, gr=None) -> torch.Tensor:
    """Mlp.forward, [V]:55-62."""
    if gr is None:
        hdn = r(gelu_erf(xn @ r(P[pre + "fc1.weight"]).t() + P[pre + "fc1.bias"]))
        return hdn @ r(P[pre + "fc2.weight"]).t() + P[pre + "fc2.bias"]
    hpre = gr(gr(xn) @ r(P[pre + "fc1.weight"]).t() + P[pre + "fc1.bias"])
    hdn = r(_GeluSavedBf16.apply(hpre))
    return gr(hdn @ r(P[pre + "fc2.weight"]).t() + P[pre + "fc2.bias"])


def conv_transpose_2x2(x: torch.Tensor, w: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """ConvTranspose2d(k=2, s=2): out[b,co,2y+dy,2x+dx] = sum_ci x[b,ci,y,x] W[ci,co,dy,dx] + b[co]  ([V]:642)."""
    B, Ci, H, W = x.shape
    Co = w.shape[1]
    o = torch.einsum("biyx,iokl->boykxl", x, w).reshape(B, Co, 2 * H, 2 * W)
    return o + b[None, :, None, None]


def fpn_tail(feats: List[torch.Tensor], P: Dict[str, torch.Tensor], eps: float, r=_ident, gr=None) -> List[torch.Tensor]:
    """fpn1..fpn4 for patch_size 16 ([V]:640-654,807-811); Norm2d = LN over channels ([V]:576-584)."""
    g_ = gr if gr is not None else _ident
    f1 = g_(r(conv_transpose_2x2(r(feats[0]), r(P["fpn1.0.weight"]), P["fpn1.0.bias"])))
    f1 = layer_norm(f1.permute(0, 2, 3, 1), P["fpn1.1.ln.weight"], P["fpn1.1.ln.bias"], eps).permute(0, 3, 1, 2)
    f1 = g_(r(conv_transpose_2x2(g_(r(gelu_erf(f1))), r(P["fpn1.3.weight"]), P["fpn1.3.bias"])))
    f2 = g_(r(conv_transpose_2x2(r(feats[1]), r(P["fpn2.0.weight"]), P["fpn2.0.bias"])))
    f3 = feats[2]
    B, C, H, W = feats[3].shape
    f4 = feats[3][:, :, :H // 2 * 2, :W // 2 * 2].reshape(B, C, H // 2, 2, W // 2, 2).amax(dim=(3, 5))
    return [f1.contiguous(), f2.contiguous(), f3.contiguous(), f4.contiguous()]


# ----------------------------------------------------------------------------------------------
# the model
# ----------------------------------------------------------------------------------------------

def backbone_forward(P: Dict[str, torch.Tensor], cfg: OracleConfig, x: torch.Tensor,
                     keep: Optional[torch.Tensor] = None) -> List[torch.Tensor]:
    """ViT_Win_RVSA_V3_WSZ7.forward ([V]:787-817).

    keep: optional (depth, 2, B) DropPath multipliers (``bernoulli(keep_p)/keep_p`` per sample, one draw for the
    attention branch and one for the MLP branch of each block, timm ``drop_path`` semantics, [V]:31-39,508-509).
    ``None`` = eval mode.
    """
    B = x.shape[0]
    hp = wp = None
    C, nH = cfg.embed_dim, cfg.num_heads
    r = _ste_bf16 if cfg.emulate_bf16 else _ident
    gr = _round_grad if (cfg.emulate_bf16 and cfg.emulate_bf16_grad) else None
    g_ = gr if gr is not None else _ident
    t = g_(patch_embed(r(x), r(P["patch_embed.proj.weight"]), P["patch_embed.proj.bias"], cfg.patch_size))
    hp, wp = x.shape[2] // cfg.patch_size, x.shape[3] // cfg.patch_size
    if "pos_embed" in P:
        t = t + P["pos_embed"]                                                   # [V]:793-794
    feats = []
    for i in range(cfg.depth):
        pre = f"blocks.{i}."
        xn = r(layer_norm(t, P[pre + "norm1.weight"], P[pre + "norm1.bias"], cfg.ln_eps))
        if cfg.is_window_block(i):
            a = rvsa_attention(xn, P, pre + "attn.", hp, wp, nH, r, gr)
        else:
            a = full_attention(xn, P, pre + "attn.", hp, wp, nH, cfg.full_attn_rel_pos, r, gr)
        if keep is not None:
            a = a * keep[i, 0].reshape(B, 1, 1)
        t = t + a                                                                # [V]:508
        xn = r(layer_norm(t, P[pre + "norm2.weight"], P[pre + "norm2.bias"], cfg.ln_eps))
        m = mlp(xn, P, pre + "mlp.", r, gr)
        if keep is not None:
            m = m * keep[i, 1].reshape(B, 1, 1)
        t = t + m                                                                # [V]:509
        if cfg.feature_mode == "multi" and i in cfg.out_indices:
            feats.append(t)
    if cfg.feature_mode == "last_norm":                                          # mmdet RVSA_MTP twin (SURVEY §2.2)
        last = r(layer_norm(t, P["norm.weight"], P["norm.bias"], cfg.ln_eps))
        feats = [last, last, last, last]
    feats = [f.permute(0, 2, 1).reshape(B, C, hp, wp) for f in feats]            # [V]:807
    if cfg.apply_fpn:
        return fpn_tail(feats, P, cfg.ln_eps, r, gr)
    return [f.contiguous() for f in feats]


def synthetic_loss(feats: Sequence[torch.Tensor]) -> torch.Tensor:
    """Stand-in objective for fwd+bwd parity and the bench (SURVEY.md §8d C2): sum of per-map means of squares/2.

    Chosen over a plain mean so the gradient depends on the activations (a plain mean gives a constant cotangent)."""
    return sum((f.float() ** 2).mean() * 0.5 for f in feats)


def algorithmic_gflop_per_image(cfg: OracleConfig) -> Dict[str, float]:
    """SURVEY.md Appendix C formulas (2*M*N*K convention, un-padded 49-token windows). Forward, per image."""
    C, nH, d = cfg.embed_dim, cfg.num_heads, cfg.depth
    hd = C // nH
    g = cfg.grid
    N = g * g
    pt, pb, pl, pr = window_padding(g, g)
    nwin = ((g + pt + pb) // WS) * ((g + pl + pr) // WS)
    n_win_blocks = sum(1 for i in range(d) if cfg.is_window_block(i))
    n_full = d - n_win_blocks
    hid = int(C * cfg.mlp_ratio)
    out = {
        "qkv": 2.0 * N * C * 3 * C * d, "proj": 2.0 * N * C * C * d,
        "fc1": 2.0 * N * C * hid * d, "fc2": 2.0 * N * hid * C * d,
        "win_qk_av": n_win_blocks * nwin * nH * 4.0 * 49 * 49 * hd,
        "win_relpos": n_win_blocks * nwin * nH * 4.0 * 49 * 7 * hd,
        "grid_sample": n_win_blocks * nwin * nH * 2.0 * 49 * hd * 8,
        "full_qk_av": n_full * nH * 4.0 * N * N * hd,
        "full_relpos": n_full * nH * 4.0 * N * g * hd if cfg.full_attn_rel_pos else 0.0,
        "patch": 2.0 * N * (cfg.in_chans * cfg.patch_size ** 2) * C,
        "fpn": 2.0 * N * C * 4 * C * (1 + 4 + 1) if cfg.apply_fpn else 0.0,
    }
    out = {k: v / 1e9 for k, v in out.items()}
    out["attn_mlp"] = sum(out[k] for k in ("qkv", "proj", "fc1", "fc2", "win_qk_av", "win_relpos", "full_qk_av", "full_relpos"))
    out["total"] = sum(v for k, v in out.items() if k != "attn_mlp")
    return out
