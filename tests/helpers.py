"""Shared test utilities: golden fixture loading and oracle plumbing (tests only)."""
import dataclasses
import hashlib
import os
import statistics
import zlib

import numpy as np
import torch

from oracle import rvsa_oracle as O

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
MAP_SAMPLES = 512        # output-map entries kept per map in reference_pinning.npz
TINY_MAP_SAMPLES = 4096  # ... and in tiny160.npz / tiny224.npz, whose sampled rel-L2 the GPU parity tests bound


# ---- hashed test data: weights and inputs are a pure function of (seed, name, position) computed in integer arithmetic, so the fixtures
#      taken from the original project need not store them and every machine regenerates them bit for bit
def hash_uniform(n, seed):
    """n float32 values in [0, 1): splitmix64 of (seed, index), top 24 bits."""
    z = np.arange(n, dtype=np.uint64) + np.array([seed], dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15)
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    z = z ^ (z >> np.uint64(31))
    return (z >> np.uint64(40)).astype(np.float32) / np.float32(2 ** 24)


def hashed_tensor(shape, seed, name, std=1.0, mean=0.0):
    """Uniform values of the given standard deviation and mean."""
    u = hash_uniform(int(np.prod(shape)), (seed << 32) | zlib.crc32(name.encode()))
    return torch.from_numpy((u * np.float32(2) - np.float32(1)) * np.float32(std * 3 ** 0.5) + np.float32(mean)).reshape(shape)


def hashed_state_dict(template, seed):
    """Weights for every floating-point entry of ``template`` (any state_dict of the backbone), at the scales of the reference's
    initialisation: LayerNorm scales 1 +- 0.02, sampling heads ~ 4x a default Conv2d init, everything else std 0.02.  Integer
    buffers are taken from ``template``."""
    C = template["pos_embed"].shape[-1]
    out = {}
    for k, v in template.items():
        if not v.is_floating_point():
            out[k] = v.clone()
        elif k.endswith(".weight") and v.ndim == 1:
            out[k] = hashed_tensor(v.shape, seed, k, 0.02, 1.0)
        else:
            out[k] = hashed_tensor(v.shape, seed, k, 4.0 / (3 * C) ** 0.5 if ".sampling_" in k else 0.02)
    return out


def sample_points(n, k=MAP_SAMPLES):
    """k distinct, evenly scattered flat indices into n entries (a Weyl sequence with a prime step)."""
    return torch.from_numpy(((np.arange(min(n, k), dtype=np.uint64) * np.uint64(2654435761)) % np.uint64(n)).astype(np.int64))


def map_summary(o, k=MAP_SAMPLES):
    """What the fixtures keep of an output map: its shape, k entries (sample_points) and its per-channel means (float64)."""
    return {"shape": np.array(o.shape, dtype=np.int64), "samples": o.reshape(-1)[sample_points(o.numel(), k)].numpy(),
            "chmean": o.double().transpose(0, 1).reshape(o.shape[1], -1).mean(1).numpy()}


def _map_refs(z, prefix, n_outs):
    assert n_outs == sum(1 for k in z.files if k.startswith(prefix + "/out") and k.endswith("/shape"))
    return [{f: z[f"{prefix}/out{i}/{f}"] for f in ("shape", "samples", "chmean")} for i in range(n_outs)]


def check_maps(outs, z, prefix, tol):
    """Every sampled entry and every channel mean of ``outs`` within ``tol`` of the stored reference values."""
    for i, (o, ref) in enumerate(zip(outs, _map_refs(z, prefix, len(outs)))):
        o = o.detach().cpu()
        assert tuple(o.shape) == tuple(ref["shape"]), (prefix, i, tuple(o.shape))
        got = map_summary(o, len(ref["samples"]))
        assert float(np.abs(got["samples"] - ref["samples"]).max()) < tol, (prefix, i)
        assert float(np.abs(got["chmean"] - ref["chmean"]).max()) < tol, (prefix, i)


def sampled_rel_l2(outs, z, prefix):
    """Per map: shape check, then the relative L2 distance of the stored sample of entries from the reference's."""
    errs = []
    for i, (o, ref) in enumerate(zip(outs, _map_refs(z, prefix, len(outs)))):
        o = o.detach().float().cpu()
        assert tuple(o.shape) == tuple(ref["shape"]), (prefix, i, tuple(o.shape))
        got = o.reshape(-1)[sample_points(o.numel(), len(ref["samples"]))].double()
        want = torch.from_numpy(ref["samples"]).double()
        errs.append(float((got - want).norm() / want.norm().clamp_min(1e-30)))
    return errs


def tensor_sha256(t):
    return hashlib.sha256(t.detach().contiguous().cpu().numpy().tobytes()).hexdigest()


GOLDEN_CFGS = {
    "tiny160": dict(img_size=160, embed_dim=128, depth=4, num_heads=2, interval=2, out_indices=(0, 1, 2, 3)),
    "tiny224": dict(img_size=224, embed_dim=128, depth=4, num_heads=2, interval=2, out_indices=(0, 1, 2, 3)),
}
GRAD_SAMPLES = 256

# ---- self-calibrating full-model parity criterion ------------------------------------------------------------------------
FWD_RATIO = 1.5          # forward maps: cuda-vs-fp32 error / emulation-vs-fp32 error
GRAD_RATIO = 2.0         # per parameter gradient
GRAD_RATIO_MEDIAN = 1.3  # over all (non coordinate-sensitive) gradients
GRAD_FLOOR = 2e-3        # absolute rel-L2 slack for gradients whose bf16 error is tiny
COORD_SENSITIVE_MAX = 0.6   # sampling-head gradients are piecewise constant in the sample coordinates (DESIGN 5): sanity bound only


def build_backbone(embed_dim, depth, num_heads, interval, out_indices, seed, img_size=224):
    from mtp_b200 import ViT_Win_RVSA_V3_WSZ7
    torch.manual_seed(seed)
    m = ViT_Win_RVSA_V3_WSZ7(img_size=img_size, patch_size=16, embed_dim=embed_dim, depth=depth, num_heads=num_heads, mlp_ratio=4, qkv_bias=True,
                             use_abs_pos_emb=True, interval=interval, out_indices=out_indices, drop_path_rate=0.1, use_rel_pos_bias=True)
    with torch.no_grad():
        for n, p in m.named_parameters():
            if "rel_pos" in n:                   # the reference initialises these tables to zero; make them count
                p.normal_(0, 0.02)
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    return m, sd


def _rel(a, b):
    a = a.detach().float().cpu()
    b = b.detach().float().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def _oracle_run(sd, cfg, x, keep, grads=True):
    P = {k: (v.clone().requires_grad_(grads) if v.is_floating_point() else v) for k, v in sd.items()}
    with torch.set_grad_enabled(grads):
        outs = O.backbone_forward(P, cfg, x, keep=keep)
        if grads:
            O.synthetic_loss(outs).backward()
    return [o.detach() for o in outs], {k: v.grad for k, v in P.items() if v.is_floating_point() and v.grad is not None}


def _coordinate_sensitive(name, cfg):
    if ".attn.sampling_" in name:
        return True
    return any(name.startswith(f"blocks.{i}.norm1.") for i in range(cfg.depth) if cfg.is_window_block(i))


def parity_check(tag, m, outs, sd, cfg, x, keep, backward=True, direct=None):
    """Self-calibrating parity criterion (see tests/test_zz_fullsize_gpu.py).  ``direct=(fwd_tol, grad_tol)``: for shallow models, where
    two bf16 implementations have not decorrelated yet, additionally bound cuda-vs-emulation directly."""
    o32, g32 = _oracle_run(sd, cfg, x, keep, grads=backward)
    o16, g16 = _oracle_run(sd, dataclasses.replace(cfg, emulate_bf16=True, emulate_bf16_grad=True), x, keep, grads=backward)
    e_cuda = [_rel(o, r) for o, r in zip(outs, o32)]
    e_emul = [_rel(o, r) for o, r in zip(o16, o32)]
    e_pair = [_rel(o, r) for o, r in zip(outs, o16)]
    print(f"{tag} forward rel-L2 per map: cuda-vs-fp32 {['%.2e' % e for e in e_cuda]}  emulation-vs-fp32 {['%.2e' % e for e in e_emul]}"
          f"  cuda-vs-emulation {['%.2e' % e for e in e_pair]}")
    for k, (ec, ee) in enumerate(zip(e_cuda, e_emul)):
        assert ec <= FWD_RATIO * ee, f"{tag}: map {k}: cuda-vs-fp32 {ec:.3e} > {FWD_RATIO} x bf16 error level {ee:.3e}"
    if direct is not None:
        assert max(e_pair) <= direct[0], f"{tag}: forward cuda-vs-emulation {e_pair}"
    if not backward:
        return
    ratios, rows = [], []
    for name, p in m.named_parameters():
        if name not in g32:
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, f"{name} should receive no gradient"
            continue
        assert p.grad is not None, f"{tag}: no gradient for {name}"
        ec, ee = _rel(p.grad, g32[name]), _rel(g16[name], g32[name])
        assert ec == ec, f"{tag}: NaN gradient for {name}"
        if _coordinate_sensitive(name, cfg):
            assert ec <= max(COORD_SENSITIVE_MAX, 3.0 * ee), f"{tag}: {name}: {ec:.3e} (emulation {ee:.3e})"
            continue
        rows.append((name, ec, ee))
        if direct is not None:
            ed = _rel(p.grad, g16[name])
            assert ed <= direct[1], f"{tag}: {name}: cuda-vs-emulation {ed:.3e}"
        ratios.append(ec / max(ee, 1e-12))
        assert ec <= GRAD_RATIO * ee + GRAD_FLOOR, f"{tag}: {name}: cuda-vs-fp32 {ec:.3e} > {GRAD_RATIO} x bf16 error level {ee:.3e}"
    rows.sort(key=lambda r: -r[1])
    med = statistics.median(ratios)
    print(f"{tag} gradients: {len(rows)} tensors, ratio cuda/emulation median {med:.2f} max {max(ratios):.2f}; largest cuda-vs-fp32:",
          [(k, "%.2e" % a, "%.2e" % b) for k, a, b in rows[:5]])
    assert med <= GRAD_RATIO_MEDIAN, f"{tag}: median error ratio {med:.2f}"


def golden_inputs(name, batch):
    """The weights and the input the reference ran with for fixture ``name``: the reference's own initialisation under
    torch.manual_seed(0), which the drop-in class reproduces bit for bit (tests/golden/make_golden.py checks it), with the re-draws
    of oracle/ref_import.build_reference; the input is torch.randn under torch.manual_seed(1234).  The global RNG is left alone."""
    from mtp_b200 import ViT_Win_RVSA_V3_WSZ7
    c = GOLDEN_CFGS[name]
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(0)
        m = ViT_Win_RVSA_V3_WSZ7(img_size=c["img_size"], patch_size=16, embed_dim=c["embed_dim"], depth=c["depth"], num_heads=c["num_heads"],
                                 mlp_ratio=4, qkv_bias=True, use_abs_pos_emb=True, interval=c["interval"], out_indices=list(c["out_indices"]),
                                 drop_path_rate=0.1, use_rel_pos_bias=True)
        g = torch.Generator().manual_seed(1)
        with torch.no_grad():
            for n, p in m.named_parameters():
                if "rel_pos" in n:
                    p.copy_(torch.randn(p.shape, generator=g) * 0.02)
                elif "sampling_" in n:
                    p.mul_(4.0)
                elif n.endswith(".bias") or "norm" in n or ".ln." in n:
                    p.add_(torch.randn(p.shape, generator=g) * 0.02)
        torch.manual_seed(1234)
        x = torch.randn(batch, 3, c["img_size"], c["img_size"])
    return {k: v.detach().clone() for k, v in m.state_dict().items()}, x


def load_golden(name):
    """Fixture ``name`` (tests/golden/make_golden.py): "sd" / "x" regenerated (golden_inputs, checked against the stored norms), the
    reference's loss, its output maps as stored by map_summary ("z", prefix "fwd": check_maps / sampled_rel_l2) and its gradients
    ("gnorm", "gfull", "gsamp")."""
    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    g = {"z": z, "loss": float(z["loss"]), "gnorm": {}, "gfull": {}, "gsamp": {}}
    g["sd"], g["x"] = golden_inputs(name, int(z["batch"]))
    for k, v in list(g["sd"].items()) + [("x", g["x"])]:
        want = float(z["norm/" + k])
        assert abs(float(v.double().norm()) - want) <= 1e-6 * max(want, 1.0), \
            f"{name}: regenerated {k} is not what the reference ran with: the initialisation changed, regenerate the fixture"
    for k in z.files:
        for grp in ("gnorm", "gfull", "gsamp"):
            if k.startswith(grp + "/"):
                v = z[k]
                g[grp][k[len(grp) + 1:]] = torch.from_numpy(v) if v.ndim else float(v)
    g["cfg"] = O.OracleConfig(**GOLDEN_CFGS[name])
    return g


def sample_idx(n):
    return np.unique(np.linspace(0, n - 1, min(n, GRAD_SAMPLES)).astype(np.int64))


def rel_l2(a, b):
    a = a.double().reshape(-1)
    b = b.double().reshape(-1)
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def check_grads_against_golden(named_grads, g, tol, skip=()):
    """named_grads: dict name -> tensor (cpu).  Compares against golden norms + samples / full tensors."""
    worst = 0.0
    for k, gn in g["gnorm"].items():
        if k in skip:
            continue
        assert k in named_grads and named_grads[k] is not None, f"missing grad {k}"
        got = named_grads[k].detach().double().cpu()
        denom = max(gn, 1e-12)
        if k in g["gfull"]:
            ref = g["gfull"][k].double()
            err = float((got - ref).norm()) / denom
        else:
            ref = g["gsamp"][k].double()
            flat = got.reshape(-1)
            idx = torch.from_numpy(sample_idx(flat.numel()))
            # sampled entries: scale the error to the whole-tensor norm via the sampling fraction
            err = float((flat[idx] - ref).norm()) / max(float(ref.norm()), 1e-12 * denom + 1e-30)
            nerr = abs(float(got.norm()) - gn) / denom
            err = max(err, nerr)
        worst = max(worst, err)
        assert err <= tol, f"grad {k}: rel err {err:.3e} > {tol:.1e}"
    return worst
