"""Worker of tests/test_gpu_loss_scaler.py's two-GPU test (one process per GPU, launched by torch.distributed.run): with a
device loss scaler, an overflow on ONE rank makes every rank skip the boundary, and all ranks keep one scale, one growth
tracker and identical parameters -- through the fused NVLink-multicast exchange and through NCCL, with no extra
communication for the scaler."""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from pairwise_sample_optimization_b200 import amp, lora  # noqa: E402
from tests._exchange_worker import make_model  # noqa: E402


def _agree(world, tensors, what):
    for t in tensors:
        gathered = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(gathered, t)
        assert all(torch.equal(gathered[0], x) for x in gathered), f"{what}: ranks disagree"


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    for fused in (True, False):
        for bits in (32, 8):
            sc = amp.DeviceGradScaler(dev, init_scale=2.0 ** 12, growth_interval=2)
            opt = lora.FusedLoRAOptimizer(make_model(dev, 8), lr=1e-3, max_grad_norm=0.5, grad_scaler=sc, optim_bits=bits,
                                          min_8bit_size=1024, exchange=lora.SymmetricGradExchange() if fused else None)
            n = opt.bucket.flat.numel()
            for boundary in range(5):
                g = torch.Generator(device=dev).manual_seed(100 * boundary + rank)
                opt.bucket.flat.copy_(torch.randn(n, device=dev, generator=g) * (1.0 + rank) * sc.scale_tensor)
                if boundary == 2 and rank == 1:
                    opt.bucket.flat[n // 2] = float("inf")
                before = opt.flat_param.clone()
                opt.all_reduce()
                opt.step()
                skipped = float(opt.found_inf) == 1.0
                assert skipped == (boundary == 2), f"rank {rank} boundary {boundary}: skip {skipped}"
                if skipped:
                    assert torch.equal(opt.flat_param, before)
                _agree(world, (opt.flat_param, sc.scale_tensor, sc.growth_tracker, opt.step_dev), f"boundary {boundary}")
                torch.cuda.synchronize()
            assert sc.get_scale() == 2.0 ** 13  # grew at boundary 1, backed off at 2, grew again at 4
            if rank == 0:
                print(f"loss scaler exchange ok: world {world}, {'multicast' if fused else 'NCCL'}, {bits}-bit", flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
