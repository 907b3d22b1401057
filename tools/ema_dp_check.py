"""Weight EMA under data parallelism with the sharded optimizer (NCCL, deferred parameter all-gathers).

    python -m torch.distributed.run --nproc-per-node 2 tools/ema_dp_check.py

Trains the small test network for 3 steps (every rank its own batch) with ema_decay = 0.9 and checks:
- after gather_state(), the full EMA is identical on every rank;
- it matches the recurrence ema += (1 - beta_k) (p - ema) over the gathered parameters, recomputed in float64, to 1e-6;
- inside ema_weights(), every rank's flat parameter buffer equals that EMA;
- after the context, every rank's flat buffer equals the live parameters bit for bit.
Exits non-zero if a check fails."""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "diffusion-deconvolution-dia-msms-data_b200"))

from dquartic.model.model import DDIMDiffusionModel  # noqa: E402
from dquartic.model.model_interface import FusedAdamW  # noqa: E402
from dquartic.model.unet1d import UNet1d  # noqa: E402

DECAY = 0.9


def same_on_all_ranks(x):
    parts = [torch.empty_like(x) for _ in range(dist.get_world_size())]
    dist.all_gather(parts, x.contiguous())
    return all(torch.equal(parts[0], q) for q in parts[1:])


def main():
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group(backend="nccl", device_id=dev)
    rank, world = dist.get_rank(), dist.get_world_size()
    torch.manual_seed(0)
    net = UNet1d(dim=4, channels=1, dim_mults=(1, 2, 2, 3, 3, 4, 4), conditional=True, init_cond_channels=1,
                 attn_cond_channels=1, downsample_dim=320, device=dev)
    dist.broadcast(net.flat_params(), src=0)
    net.mark_params_modified()
    d = DDIMDiffusionModel(net, device=dev)
    d.ema_decay = DECAY
    d._prepare_training(1e-3)
    opt = d.optimizer
    assert isinstance(opt, FusedAdamW) and opt._shard is not None, "the sharded optimizer did not engage"
    n = net.n_trainable_flat
    ref = net.flat_params()[:n].double().clone()
    g = torch.Generator(device=dev).manual_seed(100 + rank)
    for k in range(3):
        x0 = torch.rand(2, 6, 320, device=dev, generator=g)
        c2 = 0.5 * x0 + 0.5 * torch.rand(2, 6, 320, device=dev, generator=g)
        c1 = torch.rand(2, 6, device=dev, generator=g)
        d._train_one_batch(x0, ms2_cond=c2, ms1_cond=c1)
        p = net.flat_params()[:n]                    # waits for the deferred all-gathers
        w = float(torch.tensor(1.0 - min(DECAY, (1 + k) / (10 + k)), dtype=torch.float32))   # ema_w of update k
        ref = ref + w * (p.double() - ref)
    live = net.flat_params()[:n].clone()
    opt.gather_state()
    ema = opt.ema_state_dict()                       # reference format, from the gathered EMA
    full = opt._full_ema().clone()
    checks = {}
    checks["full EMA identical on every rank"] = same_on_all_ranks(full)
    err = float((full.double() - ref).abs().max() / ref.abs().max())
    checks[f"EMA vs float64 recurrence over the gathered parameters (rel {err:.2e}) < 1e-6"] = err < 1e-6
    with d.ema_weights():
        inside = net.flat_params()[:n].clone()
        sd = net.state_dict()
    checks["inside ema_weights(): flat buffer == EMA"] = torch.equal(inside, full)
    checks["inside ema_weights(): state_dict == ema_state_dict"] = all(torch.equal(sd[k], v) for k, v in ema.items())
    checks["after ema_weights(): flat buffer == live parameters"] = torch.equal(net.flat_params()[:n], live)
    checks["live parameters identical on every rank"] = same_on_all_ranks(live)
    ok = torch.tensor([int(all(checks.values()))], device=dev)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    for r in range(world):
        if r == rank:
            for name, good in checks.items():
                print(f"rank {rank}/{world} {'ok  ' if good else 'FAIL'} {name}", flush=True)
        dist.barrier()
    if rank == 0:
        print(f"{torch.cuda.get_device_name(dev)} x {world}: {'PASS' if int(ok) else 'FAIL'}", flush=True)
    dist.destroy_process_group()
    sys.exit(0 if int(ok) else 1)


if __name__ == "__main__":
    main()
