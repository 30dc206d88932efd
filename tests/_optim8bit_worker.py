"""Worker of tests/test_gpu_optim8bit.py's two-GPU test (one process per GPU, launched by torch.distributed.run): the fused
NVLink-multicast exchange feeding the 8-bit optimizer boundary leaves bitwise-identical codes and parameters on every rank."""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from pairwise_sample_optimization_b200 import lora  # noqa: E402
from tests._exchange_worker import make_model  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    for r in (8, 12):  # 12: operand copies with a padded pitch
        opt = lora.FusedLoRAOptimizer(make_model(dev, r), lr=1e-3, max_grad_norm=0.5, exchange=lora.SymmetricGradExchange(),
                                      optim_bits=8, min_8bit_size=1024)
        assert opt.blocks8.shape[0] > 0 and opt.chunks32.shape[0] > 0
        n = opt.bucket.flat.numel()
        for boundary in range(3):
            g = torch.Generator(device=dev).manual_seed(100 * boundary + rank)
            opt.bucket.flat.copy_(torch.randn(n, device=dev, generator=g) * (1.0 + rank))
            opt.all_reduce()
            opt.step()
            assert float(opt.bucket.flat.abs().max()) == 0.0
            for t in (opt.flat_param, opt.code1, opt.code2, opt.absmax1, opt.exp_avg32):
                gathered = [torch.empty_like(t) for _ in range(world)]
                dist.all_gather(gathered, t)
                assert all(torch.equal(gathered[0], x) for x in gathered), f"boundary {boundary}: ranks disagree"
            torch.cuda.synchronize()
        if rank == 0:
            print(f"8-bit exchange ok: world {world}, rank-{r} adapters, {opt.blocks8.shape[0]} 8-bit blocks", flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
