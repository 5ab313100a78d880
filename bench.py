#!/usr/bin/env python
"""Benchmark of the hot path: ViT + RVSA backbone pretrain step, bf16, synthetic data (BASELINE.json metric and configs).

    python bench.py --gpus 1 --steps 20 --warmup 5                      # headline: config c3 (ViT-L @224^2, 8 images per GPU)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...
    python bench.py --impl reference ...                                # the reference's CPU path (oracle port) on the host cores
    python bench.py --config c2|c4|c5 ...                               # the other BASELINE.json configurations (see CONFIGS)
    python bench.py ... --dump-outputs DIR                              # also write what the last timed step computed, DIR/<name>.npy

Headline step (c3, Multi-Task_Pretrain/models.py:306-335 + main_pretrain.py:701-832 for the encoder): three uint8 image streams
(3 + 3 + 2 images per GPU) -> MTP_DataPreprocessor arithmetic fused into the patch gather -> ONE encoder call on the concatenated
batch -> feature maps split 3|3|2 to three stand-in heads (the decoders are third-party, out of scope) -> full backward ->
gradient all-reduce (N > 1) -> global-norm clip -> fused AdamW.  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark leaves the tree it runs from as it found it (it may be read-only)

import torch  # noqa: E402

VIT = {"b": dict(embed_dim=768, depth=12, num_heads=12, interval=3, out_indices=[3, 5, 7, 11]),
       "l": dict(embed_dim=1024, depth=24, num_heads=16, interval=6, out_indices=[7, 11, 15, 23])}
# BASELINE.json `configs` (SURVEY.md 8d): model, image side, images per GPU, what a step is
CONFIGS = {
    "c2": dict(model="b", img=224, batch=32, mode="fwdbwd",
               metric="images/sec ViT-B+RVSA backbone fwd+bwd @224^2 bf16", workload="ViT-B+RVSA backbone fwd+bwd, batch 32 @224^2 (BASELINE configs[1])"),
    "c3": dict(model="l", img=224, batch=8, mode="step",
               metric="images/sec ViT-L+RVSA MTP step @224^2 bf16",
               workload="ViT-L+RVSA backbone pretrain step @224^2: 3 uint8 streams (3|3|2 img) -> fused preprocess -> one encoder call -> "
                        "3 stand-in heads -> bwd + grad all-reduce + clip + AdamW (BASELINE configs[2], 8 img/GPU)"),
    "c4": dict(model="l", img=512, batch=2, mode="step",
               metric="images/sec ViT-L+RVSA finetune-shaped step @512^2 bf16",
               workload="ViT-L+RVSA backbone step @512^2 (25 windows/img, dense blocks N=1024), 2 img/GPU, stand-in head (BASELINE configs[3])"),
    "c5": dict(model="l", img=1024, batch=1, mode="fwdbwd",
               metric="images/sec ViT-L+RVSA backbone fwd+bwd @1024^2 bf16",
               workload="ViT-L+RVSA backbone fwd+bwd @1024^2 (seq-len 4096, 100 windows/img), 1 img/GPU (BASELINE configs[4])"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--config", default="c3", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=0, help="images per GPU (0 = the config's)")
    ap.add_argument("--graph", type=int, default=1, help="capture the step into a CUDA graph")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gemm-share", action="store_true", help="skip the in-situ GEMM timing pass (leaves the training state intact)")
    ap.add_argument("--bucket-blocks", type=int, default=2, help="transformer blocks per gradient all-reduce bucket (N > 1)")
    ap.add_argument("--comm-sms", type=int, default=16, help="SMs left to NCCL while the backward runs (N > 1)")
    ap.add_argument("--grad-comm", default="bf16", choices=["bf16", "fp32"], help="dtype of the gradient all-reduce buckets (N > 1)")
    ap.add_argument("--float-input", action="store_true", help="feed a pre-normalised bf16 batch instead of uint8 + fused preprocessing")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy (float32): the loss, and "
                    "the updated parameters (step configs) or the parameter gradients (fwd+bwd configs), a fixed sample of up to 16384 entries per tensor")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs writes what the native step computed: it needs --impl native")
    return args


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback")


class ClockSampler:
    """SM clock / throttle-reason sampling (NVML) on a background thread during the timed region."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake"}

    def __init__(self, gpu_index, period=0.05):
        self.gpu, self.period, self.sm, self.reasons, self.power = gpu_index, period, [], set(), []
        self._stop = threading.Event()
        self._thr = None
        self.max_sm = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.gpu]) if vis and vis.split(",")[0].isdigit() else self.gpu
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.nv = pynvml
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()
        except Exception:
            self._thr = None

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.sm.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
                mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(self.period)

    def stop(self):
        if self._thr is None:
            return None
        self._stop.set()
        self._thr.join(timeout=1.0)
        if not self.sm:
            return None
        return {"sm_mhz": statistics.median(self.sm), "sm_max_mhz": self.max_sm, "reasons": sorted(self.reasons),
                "power_w_max": max(self.power) if self.power else None, "samples": len(self.sm)}


DUMP_PER_TENSOR = 16384       # at most 489 tensors (ViT-L) x 16384 x 4 B = 32 MB per dumped array


def dump_sample(tensors):
    """float32 concatenation, in the given order, of every tensor's entries, or of a fixed spread of DUMP_PER_TENSOR of them (a Weyl
    sequence with a prime step over the flattened tensor) when it has more.  Runs on the device; returns a host array."""
    out = []
    for t in tensors:
        f = t.detach().reshape(-1)
        if f.numel() > DUMP_PER_TENSOR:
            f = f[torch.arange(DUMP_PER_TENSOR, device=f.device) * 2654435761 % f.numel()]
        out.append(f.float())
    return torch.cat(out).cpu().numpy()


def split3(B):
    """The three task streams of models.py:327-329 (`b, b, rest`); 8 images per GPU -> 3 | 3 | 2 (SURVEY 8d C3)."""
    if B < 3:
        return None
    b = (B + 2) // 3
    return (b, b, B - 2 * b) if B - 2 * b > 0 else (b, B - b - 1, 1)


def build_module(cfg, drop_path=0.1):
    from mtp_b200 import ViT_Win_RVSA_V3_WSZ7
    v = VIT[cfg["model"]]
    torch.manual_seed(0)
    m = ViT_Win_RVSA_V3_WSZ7(img_size=cfg["img"], patch_size=16, embed_dim=v["embed_dim"], depth=v["depth"], num_heads=v["num_heads"],
                             mlp_ratio=4, qkv_bias=True, use_abs_pos_emb=True, interval=v["interval"], out_indices=v["out_indices"],
                             drop_path_rate=drop_path, use_rel_pos_bias=True)
    g = torch.Generator().manual_seed(1)
    with torch.no_grad():
        for n, p in m.named_parameters():
            if "rel_pos" in n:                      # zero-initialised in the reference: re-draw so the terms are exercised
                p.copy_(torch.randn(p.shape, generator=g) * 0.02)
    return m


def fwd_gflop_per_img(cfg):
    from oracle import rvsa_oracle as O       # formulas only (SURVEY Appendix C); nothing of the oracle is executed on the timed path
    v = VIT[cfg["model"]]
    oc = O.OracleConfig(img_size=cfg["img"], embed_dim=v["embed_dim"], depth=v["depth"], num_heads=v["num_heads"], interval=v["interval"],
                        out_indices=tuple(v["out_indices"]))
    return O.algorithmic_gflop_per_image(oc)["total"]


# ------------------------------------------------------------------------------------------------------ CPU reference arm
def usable_threads():
    """Thread count that actually maximises CPU throughput on this host.  Containers often expose every logical CPU of the
    machine while a cgroup quota / co-tenants make more than a fraction of them counter-productive (measured on the pool's
    B200 boxes: 128 logical CPUs, 16 threads are 60x faster than 128), so probe a GEMM instead of trusting cpu_count()."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(p) + 0.5)))
    except Exception:
        pass
    cands = sorted({c for c in (4, 8, 16, 32, 64, n) if c <= n})
    a = torch.randn(2048, 2048)
    times = {}
    for c in cands:
        torch.set_num_threads(c)
        a @ a
        t0 = time.perf_counter()
        for _ in range(4):
            a @ a
        times[c] = time.perf_counter() - t0
    tmin = min(times.values())
    return max(c for c in cands if times[c] <= 1.15 * tmin)      # the largest count that is still (nearly) the fastest


def cpu_reference(cfg, steps, warmup, batch, threads=None, forward_only=False):
    """The reference's CPU path (oracle port of [V], fp32, pinned to the live reference by tests/test_oracle_vs_reference.py) doing the
    same work on a bounded sample: forward + stand-in heads + backward (+ clip + AdamW for the `step` configs)."""
    from oracle import rvsa_oracle as O
    threads = threads or usable_threads()
    torch.set_num_threads(threads)
    v = VIT[cfg["model"]]
    oc = O.OracleConfig(img_size=cfg["img"], embed_dim=v["embed_dim"], depth=v["depth"], num_heads=v["num_heads"], interval=v["interval"],
                        out_indices=tuple(v["out_indices"]))
    m = build_module(cfg)
    P = {k: (v_.detach().clone().requires_grad_(not forward_only) if v_.is_floating_point() else v_) for k, v_ in m.state_dict().items()}
    del m
    params = [t for t in P.values() if t.is_floating_point()]
    opt = torch.optim.AdamW(params, lr=6e-5, weight_decay=0.05) if (cfg["mode"] == "step" and not forward_only) else None
    x = torch.randn(batch, 3, cfg["img"], cfg["img"])
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        if forward_only:
            with torch.no_grad():
                O.backbone_forward(P, oc, x)
        else:
            for p in params:
                p.grad = None
            loss = O.synthetic_loss(O.backbone_forward(P, oc, x))
            loss.backward()
            if opt is not None:
                torch.nn.utils.clip_grad_norm_([p for p in params if p.grad is not None], 5.0)
                opt.step()
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    return batch / statistics.median(times), threads, sum(times)


def cpu_sample_batch(cfg):
    return {"c2": 2, "c3": 2, "c4": 1, "c5": 1}[cfg["name"]]       # SURVEY 8d: fwd+bwd B=2 @224^2; one image at the larger sizes


def run_reference(args, cfg, rank):
    if rank != 0:
        return
    b = cpu_sample_batch(cfg)
    steps, warmup = args.steps, min(args.warmup, 2)          # ~1 s of CPU work per step (c3; SURVEY 8d asks for >= 1 warm-up + 3 timed)
    rate, threads, total = cpu_reference(cfg, steps, warmup, b)
    ms = 1000.0 * b / rate
    what = "fwd+bwd+clip+AdamW" if cfg["mode"] == "step" else "fwd+bwd"
    sample = f"{b} image(s) per step x {steps} timed steps (+{warmup} warm-up), {what}, fp32, {threads} threads, {total:.1f} s"
    line = {"impl": "reference", "metric": cfg["metric"], "value": rate, "unit": "images/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
            "config": {"workload": cfg["workload"], "implementation": "oracle port of the reference ([V]) on the host cores, fp32",
                       "per_step_batch": b},
            "cpu_baseline": {"value": rate, "unit": "images/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": rate, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------ native arm
class FwdBwdStep:
    """Configs c2 / c5: backbone forward + stand-in heads + full backward, no optimizer (BASELINE: "backbone fwd+bwd")."""

    def __init__(self, model, heads, use_cuda_graph):
        from mtp_b200 import engine, engine_bwd
        self.m, self.heads, self.use_graph = model, heads, use_cuda_graph
        self.engine, self.engine_bwd = engine, engine_bwd
        self.G = engine_bwd.GradStore(model, next(model.parameters()).device)
        self.graph = None
        self.dev = next(model.parameters()).device

    def _body(self, x):
        keep = self.engine._draw_keep(self.m, x.shape[0], x.device)
        outs, ctx = self.engine._forward_impl(self.m, x, keep, save=True)
        loss, douts = self.heads(outs)
        self.G.flat.zero_()
        self.G.touched = set()
        self.engine_bwd.backward_impl(self.m, x, ctx, douts, grad_store=self.G)
        return loss

    def step(self, x):
        if not self.use_graph:
            return self._body(x)
        if self.graph is None:
            self._x = x.clone()
            s = torch.cuda.Stream(device=self.dev)
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                for _ in range(2):
                    self._body(self._x)
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self._loss = self._body(self._x)
        if x.data_ptr() != self._x.data_ptr():
            self._x.copy_(x, non_blocking=True)
        self.graph.replay()
        return self._loss

    def step_from_host(self, parts):
        if isinstance(parts, (tuple, list)):
            x = torch.cat([p.to(self.dev, non_blocking=True) for p in parts], 0)
        else:
            x = parts.to(self.dev, non_blocking=True)
        return float(self.step(x).item())

    def _step_body(self, x):
        return self._body(x)


def gemm_flops_and_bytes(runner, x):
    """One eager (non-graph) step with every GEMM launch recorded: count, 2*M*N*K, algorithmic bytes (operands read once +
    outputs written once)."""
    from mtp_b200 import ops
    tot = dict(n=0, flops=0.0, bytes=0.0)
    orig, orig_dual = ops.gemm, ops.gemm_dual

    def alg_bytes(M, N, K, out, aux=None, out2=None, **_):
        b = 2.0 * (M * K + N * K) + out.element_size() * M * N
        if aux is not None:
            b += aux.element_size() * M * N
        if out2 is not None:
            b += out2.element_size() * M * N
        return b

    def rec(A, B, M, N, K, out, **kw):
        tot["n"] += 1
        tot["flops"] += 2.0 * M * N * K
        tot["bytes"] += alg_bytes(M, N, K, out, aux=kw.get("aux"), out2=kw.get("out2"))
        return orig(A, B, M, N, K, out, **kw)

    def rec_dual(g0, g1, force_bn=0):
        tot["n"] += 1
        for g in (g0, g1):
            tot["flops"] += 2.0 * g["M"] * g["N"] * g["K"]
            tot["bytes"] += alg_bytes(g["M"], g["N"], g["K"], g["out"], aux=g.get("aux"), out2=g.get("out2"))
        return orig_dual(g0, g1, force_bn)
    ops.gemm, ops.gemm_dual = rec, rec_dual
    try:
        runner._step_body(x)
        torch.cuda.synchronize()
    finally:
        ops.gemm, ops.gemm_dual = orig, orig_dual
    return tot


def count_launches(runner, x):
    """Kernels of libmtp_b200.so launched per step (entry point -> kernels it enqueues)."""
    from mtp_b200 import _lib
    per_call = {"mtp_rvsa_attn_bwd": 3}          # attention backward + partial reduce + kv finalize (the memset is not a kernel of ours)
    n = [0]
    orig = _lib.call

    def counting(name, *a):
        if not name.startswith(("mtp_set_", "mtp_gemm_set_", "mtp_gemm_last", "mtp_gemm_plan")):
            n[0] += per_call.get(name, 1)
        return orig(name, *a)
    _lib.call = counting           # ops / trainer / engine_bwd all call through the module attribute
    try:
        runner._step_body(x)
        torch.cuda.synchronize()
    finally:
        _lib.call = orig
    return n[0]


def main():
    args = parse()
    cfg = dict(CONFIGS[args.config], name=args.config)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, cfg, rank)
        return
    assert torch.cuda.is_available(), "bench.py (native arm) needs a CUDA device"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    import torch.distributed as dist
    if world > 1:
        if args.comm_sms > 0:
            os.environ.setdefault("NCCL_MAX_CTAS", str(args.comm_sms))       # the SMs PretrainStep(comm_sms=) leaves to the all-reduce kernels
        dist.init_process_group("nccl", device_id=dev)
    from mtp_b200 import _lib
    from mtp_b200.preprocess import ImagePreprocess
    from mtp_b200.trainer import PretrainStep, ThreeTaskHeads, synthetic_heads
    _lib.load()
    B = args.batch or cfg["batch"]
    S = cfg["img"]
    model = build_module(cfg).to(dev).train()
    u8 = not args.float_input
    if u8:
        model.input_preprocess = ImagePreprocess(out_dtype=torch.bfloat16)          # models.py:37-41 mean / std / bgr_to_rgb
    split = split3(B)
    heads = ThreeTaskHeads(split) if split else synthetic_heads
    if cfg["mode"] == "step":
        runner = PretrainStep(model, lr=6e-5, weight_decay=0.05, max_norm=5.0, t_max=80000, use_cuda_graph=bool(args.graph),
                              bucket_blocks=args.bucket_blocks, comm_sms=args.comm_sms, heads=heads, grad_comm=args.grad_comm)
    else:
        runner = FwdBwdStep(model, heads, bool(args.graph))
    g = torch.Generator().manual_seed(1234 + rank)
    sizes = list(split) if split else [B]
    if u8:
        parts_host = [torch.randint(0, 256, (b, 3, S, S), dtype=torch.uint8, generator=g).pin_memory() for b in sizes]
    else:
        parts_host = [torch.randn(b, 3, S, S, generator=g).to(torch.bfloat16).pin_memory() for b in sizes]
    x = torch.cat([p.to(dev) for p in parts_host], 0)
    h2d = sum(p.numel() * p.element_size() for p in parts_host)

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- eager instrumented passes (also serve as warm-up for kernel attributes / allocator)
    want_graph = bool(args.graph)
    runner.use_cuda_graph = False
    if hasattr(runner, "use_graph"):
        runner.use_graph = False
    for _ in range(2):
        runner.step(x)
    torch.cuda.synchronize()
    launches = count_launches(runner, x)
    gm = gemm_flops_and_bytes(runner, x)
    runner.use_cuda_graph = want_graph
    if hasattr(runner, "use_graph"):
        runner.use_graph = want_graph

    # ---- device-resident timing (inputs in HBM; the working set of a step is >> L2, see config.l2)
    W = max(3, args.warmup)
    for _ in range(W):
        loss = runner.step(x)
    sync_all()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss = runner.step(x)
    e1.record()
    sync_all()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if sampler else None
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = t.item() / args.steps
    value = world * B / (ms_step / 1e3)
    final_loss = float(loss.item())
    dump = None
    if args.dump_outputs and rank == 0:          # read now: the passes below advance (end to end) and then garble (GEMM share) the state
        if cfg["mode"] == "step":
            dump = {"loss": loss, "params": [p for _, p in model.named_parameters()]}
        else:
            dump = {"loss": loss, "grads": [runner.G.views[n] for n in runner.G.names]}
        dump = {k: dump_sample(v if isinstance(v, list) else [v]) for k, v in dump.items()}

    # ---- end to end: pinned host uint8 streams -> device -> step -> loss back on the host, every step
    for _ in range(2):
        runner.step_from_host(parts_host)
    sync_all()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        runner.step_from_host(parts_host)
    sync_all()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    t = torch.tensor([e2e_ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * B / (t.item() / args.steps / 1e3)

    # ---- GEMM time inside the graph-replayed step, measured live at every N: the same step re-captured with empty GEMM launches
    #      (mtp_gemm_set_debug_mode 4); the difference is what the tcgen05 GEMM kernels cost in situ -- launch gaps, PDL overlap and
    #      store drain included, i.e. the conservative reading.  Run last: the training state is garbage afterwards.
    gemm_ms = None
    if args.graph and not args.no_gemm_share:
        try:
            _lib.call("mtp_gemm_set_debug_mode", 4)
            runner.graph = None
            for _ in range(3):
                runner.step(x)
            sync_all()
            e0.record()
            for _ in range(args.steps):
                runner.step(x)
            e1.record()
            sync_all()
            t = torch.tensor([e0.elapsed_time(e1)], device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            gemm_ms = ms_step - t.item() / args.steps
        finally:
            _lib.call("mtp_gemm_set_debug_mode", 0)

    if rank == 0:
        pk = peaks()
        gf = fwd_gflop_per_img(cfg)
        step_tflops = 3.0 * gf * (value / world) / 1e3          # per GPU; training step = 3 x forward (SURVEY 8d)
        gemm_tflops = gm["flops"] / (gemm_ms * 1e-3) / 1e12 if gemm_ms and gemm_ms > 0 else None
        line = {
            "metric": cfg["metric"], "value": value, "unit": "images/s", "n_gpus": world,
            "steps": args.steps, "warmup": W, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": cfg["workload"], "name": args.config, "per_gpu_batch": B, "global_batch": B * world,
                       "streams": list(split) if split else [B], "input": "uint8 CHW + fused MTP_DataPreprocessor" if u8 else "bf16 normalised",
                       "tokens_per_gpu": B * (S // 16) ** 2, "parallelism": f"dp{world}",
                       "grad_allreduce": (f"{args.grad_comm} buckets of {args.bucket_blocks} blocks, pyramid weights first, small params fp32 last; "
                                          f"{args.comm_sms} SMs left to NCCL") if world > 1 else None, "cuda_graph": bool(args.graph),
                       "l2": "per-step working set (weights + activations + gradients, GBs) >> 126 MB L2; no explicit flush", "loss": final_loss},
            "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4},
            "gpu_launches": launches * args.steps,
            "roofline": {"bound": "tensor", "kernel": "gemm_bf16_kernel (all tcgen05 GEMM launches of one step)", "achieved": gemm_tflops,
                         "peak": pk["tf_burst"], "unit": "TFLOP/s", "frac": (gemm_tflops / pk["tf_burst"]) if gemm_tflops else None,
                         "traffic": None,       # DRAM bytes are not measurable from inside the run (r1 verdict: never quote a committed file here);
                         #                        the ncu pass of this command lives in profiles/ (r2_gemm_dram_final.json: 3.94 GB per step)
                         "algorithmic_bytes_per_step": gm["bytes"], "peak_source": pk["src"] + " (burst cuBLAS bf16)",
                         "gemm_launches_per_step": gm["n"], "gemm_gflop_per_step": gm["flops"] / 1e9, "gemm_ms_per_step": gemm_ms,
                         "gemm_timing": "in situ: graph-replayed step minus the same step with empty GEMM launches (all ranks, max)",
                         "gemm_share_of_step": gemm_ms / ms_step if gemm_ms else None,
                         "step_tflops_per_gpu": step_tflops, "step_frac_of_sustained_peak": step_tflops / pk["tf_sustained"]},
            "clocks": clocks,
        }
        if not args.no_cpu_baseline and world == 1:
            try:
                b = cpu_sample_batch(cfg)
                n_cpu = 8 if cfg["name"] in ("c2", "c3") else 3          # ~10 s of CPU work at 224^2; the larger inputs take seconds per step
                rate, threads, total = cpu_reference(cfg, n_cpu, 1, b)
                what = "fwd+bwd+clip+AdamW" if cfg["mode"] == "step" else "fwd+bwd"
                cb = {"value": rate, "unit": "images/s", "cores": threads, "kind": "port",
                      "sample": f"{b} images/step x {n_cpu} timed steps (+1 warm-up), {what}, fp32 oracle port of [V], {total:.1f} s"}
                if args.config == "c3":         # SURVEY 8d also asks for the forward at B = 8
                    frate, _, ftotal = cpu_reference(cfg, 3, 1, 8, threads=threads, forward_only=True)
                    cb["forward_only"] = {"value": frate, "unit": "images/s", "sample": f"8 images x 3 timed forwards (+1 warm-up), {ftotal:.1f} s"}
                line["cpu_baseline"] = cb
            except Exception as ex:      # the baseline is informative; never lose the GPU line to it
                line["cpu_baseline"] = {"error": repr(ex)}
        print(json.dumps(line), flush=True)
    if dump is not None:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in dump.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
