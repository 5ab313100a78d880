"""Data-parallel step on REAL GPUs (needs >= 2 devices): after the bucketed all-reduce the gradients of two ranks with half
the batch each equal the single-GPU gradients of the whole batch (SURVEY 4.1-8) -- exactly (fp32 rounding) with fp32 buckets, to bf16
rounding with bf16 buckets -- and one optimizer step leaves both ranks with identical parameters."""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu


def _worker(rank, world, port, grad_comm, graph, out):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), NCCL_MAX_CTAS="8")
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
    try:
        from mtp_b200.trainer import PretrainStep
        from tests.helpers import load_golden
        from tests.test_backbone_gpu import build_module
        g = load_golden("tiny160")
        x_all = torch.cat([g["x"], g["x"].flip(0) * 0.5], 0).cuda()          # 4 images
        per = x_all.shape[0] // world

        def fresh():
            m = build_module("tiny160")
            m.load_state_dict(g["sd"])
            return m.cuda().eval()
        # single-GPU reference on the whole batch: a trainer bound to a process group of this rank alone (world size 1)
        groups = [dist.new_group([r]) for r in range(world)]              # collective: every rank creates every group
        m_ref = fresh()
        ref = PretrainStep(m_ref, lr=1e-3, max_norm=0.0, process_group=groups[rank])
        assert ref.world == 1
        ref._forward_backward(x_all, lambda r: None)
        g_ref = ref.flat_g.clone()
        # data-parallel trainer on this rank's half
        m = fresh()
        tr = PretrainStep(m, lr=1e-3, max_norm=1.0, bucket_blocks=2, comm_sms=8, grad_comm=grad_comm, use_cuda_graph=graph)
        assert tr.world == world
        if not graph:
            tr._forward_backward(x_all[rank * per:(rank + 1) * per], tr._reduce)
            torch.cuda.current_stream().wait_stream(tr.comm_stream)
            torch.cuda.synchronize()
            got = tr.flat_g.clone() / world
            if grad_comm == "bf16":
                got[tr.small_end:] = tr.flat_g16[tr.small_end:].float() / world
            err = float((got - g_ref).norm() / g_ref.norm())
            worst = 0.0
            for n, o in tr.offsets.items():
                k = tr.layout.numel[n]
                den = float(g_ref[o:o + k].norm())
                if den > 0:
                    worst = max(worst, float((got[o:o + k] - g_ref[o:o + k]).norm()) / den)
            out[rank] = (err, worst)
        else:
            for _ in range(2):
                tr.step(x_all[rank * per:(rank + 1) * per])
            torch.cuda.synchronize()
            flat = tr.flat_p.clone()
            gathered = [torch.empty_like(flat) for _ in range(world)]
            dist.all_gather(gathered, flat)
            out[rank] = (float((gathered[0] - gathered[1]).abs().max()), 0.0)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("grad_comm,graph", [("fp32", False), ("bf16", False), ("bf16", True)])
def test_two_rank_gradients_equal_single_gpu(grad_comm, graph):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    out = ctx.Manager().dict()
    port = 29600 + (hash((grad_comm, graph)) % 200)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, grad_comm, graph, out)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(300)
        assert p.exitcode == 0, f"rank exited with {p.exitcode}"
    print(grad_comm, "graph" if graph else "eager", dict(out))
    for r in range(2):
        err, worst = out[r]
        if graph:
            assert err == 0.0, f"ranks diverged after two steps: max |dp| = {err}"          # same reduced gradients -> bit-identical parameters
        elif grad_comm == "fp32":
            assert err < 2e-5 and worst < 2e-4, (err, worst)
        else:
            assert err < 6e-3 and worst < 1.5e-2, (err, worst)       # one bf16 rounding per rank + a bf16 sum
