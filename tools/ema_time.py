"""Cost of the weight EMA on one GPU, on the default 1.2 B-parameter denoiser.

1. dq_adamw against dq_adamw_ema on the full 1,204,738,392-element flat buffer (16-byte aligned: the vector kernels),
   CUDA events over repeated launches, the two kernels alternated; TB/s from 28 and 36 B/param.  The 5 buffers (24 GB)
   are far larger than the L2, so every launch streams from HBM.
2. The batch-256 training step (4 micro-batches of 64, 34 x 40000 maps, as bench.py times it) with the EMA off and on:
   one network, two FusedAdamW instances (ema_decay None / 0.9999) swapped in turn, rounds alternated in one process.

Prints the card name and power limit first.  Usage: python tools/ema_time.py [--rounds R] [--steps S]"""
import argparse
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "diffusion-deconvolution-dia-msms-data_b200"))
from dquartic import _native as N  # noqa: E402

N_FLAT = 1_204_738_392
CFG = dict(dim=4, dim_mults=(1, 2, 2, 3, 3, 4, 4), downsample_dim=40000)   # bench.py's DEFAULT_CFG
RT, MZ = 34, 40000


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = f"nvidia-smi unavailable ({e})"
    return f"{name}; power limit, max SM clock: {q}"


def time_ms(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def kernels(rounds, reps=10):
    n = N_FLAT
    p, g, m, e = (torch.randn(n, device="cuda") * 0.01 for _ in range(4))
    v = torch.full((n,), 1e-4, device="cuda")
    coef = torch.tensor([1.0, 1.0], device="cuda")
    args = (coef, 1e-5, 0.9, 0.999, 1e-8, 0.01, 1e-5 / 0.1, 0.0316)
    assert all(t.data_ptr() % 16 == 0 for t in (p, g, m, v, e))
    runs = {
        "dq_adamw": (28, lambda: N.call("dq_adamw", p, g, m, v, n, *args)),
        "dq_adamw_ema": (36, lambda: N.call("dq_adamw_ema", p, g, m, v, e, n, *args, 1e-4)),
    }
    for _, f in runs.values():
        f(); f()
    torch.cuda.synchronize()
    res = {k: [] for k in runs}
    for _ in range(rounds):
        for k, (_, f) in runs.items():
            res[k].append(time_ms(f, reps))
    for k, (bpp, _) in runs.items():
        ts = res[k]
        med = statistics.median(ts)
        print(f"{k:13s} n={n}: median {med:.3f} ms = {bpp * n / med / 1e9:.2f} TB/s ({bpp} B/param); "
              f"min {min(ts):.3f} max {max(ts):.3f} ms over {rounds} rounds of {reps} launches", flush=True)
    d = statistics.median(res["dq_adamw_ema"]) - statistics.median(res["dq_adamw"])
    print(f"dq_adamw_ema - dq_adamw: {d:+.3f} ms per step (median)", flush=True)
    del p, g, m, v, e
    torch.cuda.empty_cache()


def steps(rounds, n_steps, batch=256, micro=64):
    from dquartic.model.model import DDIMDiffusionModel
    from dquartic.model.model_interface import FusedAdamW
    from dquartic.model.unet1d import UNet1d

    torch.cuda.reset_peak_memory_stats()
    torch.manual_seed(1234)
    net = UNet1d(dim=CFG["dim"], channels=1, dim_mults=CFG["dim_mults"], conditional=True, init_cond_channels=1,
                 attn_cond_channels=1, downsample_dim=CFG["downsample_dim"], simple=True, device="cuda")
    print(f"trainable flat buffer: {net.n_trainable_flat} elements", flush=True)
    d = DDIMDiffusionModel(net, device="cuda")
    d.micro_batch = micro
    d._prepare_training(1e-5)
    opts = {"ema off": d.optimizer, "ema on": FusedAdamW(net, lr=1e-5, ema_decay=0.9999)}
    x0 = torch.rand(batch, RT, MZ, device="cuda") * (torch.rand(batch, RT, MZ, device="cuda") < 0.3)
    c2 = 0.5 * x0 + 0.5 * torch.rand_like(x0) * (torch.rand_like(x0) < 0.3)
    c1 = torch.rand(batch, RT, device="cuda")
    for k, o in opts.items():   # warm-up: kernels loaded, bf16 operands and the optimizer states allocated
        d.optimizer = o
        for _ in range(2):
            d._train_one_batch(x0, ms2_cond=c2, ms1_cond=c1)
    torch.cuda.synchronize()
    print(f"peak allocated in the training steps: {torch.cuda.max_memory_allocated() / 1e9:.1f} GB (both optimizers' "
          f"states: the EMA adds {opts['ema on']._ema.numel() * 4 / 1e9:.1f} GB to a single optimizer's)", flush=True)
    res = {k: [] for k in opts}
    for r in range(rounds):
        for k, o in (opts.items() if r % 2 == 0 else reversed(list(opts.items()))):
            d.optimizer = o
            d._train_one_batch(x0, ms2_cond=c2, ms1_cond=c1)   # one untimed step after the switch
            torch.cuda.synchronize()
            res[k].append(time_ms(lambda: d._train_one_batch(x0, ms2_cond=c2, ms1_cond=c1), n_steps))
    for k, ts in res.items():
        print(f"train step {k:7s} (batch {batch}, micro-batch {micro}): median {statistics.median(ts):.1f} ms, "
              f"min {min(ts):.1f} max {max(ts):.1f} ms over {rounds} rounds of {n_steps} steps: "
              + " ".join(f"{t:.1f}" for t in ts), flush=True)
    diffs = [a - b for a, b in zip(res["ema on"], res["ema off"])]
    print(f"ema on - ema off per round: " + " ".join(f"{x:+.1f}" for x in diffs)
          + f" ms; median {statistics.median(diffs):+.2f} ms = "
          f"{100 * statistics.median(diffs) / statistics.median(res['ema off']):+.2f} %", flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--steps", type=int, default=3, help="timed training steps per round")
    ap.add_argument("--kernels-only", action="store_true")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ema_time.py measures on a CUDA device; none found")
    print(card(), flush=True)
    kernels(a.rounds)
    if not a.kernels_only:
        steps(a.rounds, a.steps)


if __name__ == "__main__":
    main()
