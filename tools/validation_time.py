"""Cost of held-out validation on one GPU, on the default denoiser (34 x 40000 maps).

1. CUDA-event time of dq_map_scores at 64 x 34 x 40000 elements (two fp32 maps: 8 B per element, 696 MB per launch,
   more than the L2, so it streams from HBM), best of 3 rounds of 20 launches; bytes/s from 8 B per element.
2. `validate` at full size: 64 windows x 10 bands = 640 forwards in chunks of 64, host clock around calls that end in a
   device synchronise; forwards/s.
3. Training epochs on the 520-slice synthetic pool at batch 256 (the bench's workload), 3 steps each, without and with
   a 10 % held-out split plus `validate` after the epoch, alternated in one process; the difference is the cost of
   validation per epoch.
4. `cli.evaluate_model` (what `dquartic evaluate` runs per set of weights): `validate` plus dpm++2m@20 sampling and
   scoring of the 64 windows.

Weights: the network's seeded initialisation (speed does not depend on them).  Prints the card name and power limit
first.  Usage: python tools/validation_time.py [--rounds R]"""
import argparse
import os
import random
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "diffusion-deconvolution-dia-msms-data_b200"))
from dquartic import _native as N  # noqa: E402
from dquartic import cli  # noqa: E402
from dquartic.model.model import DDIMDiffusionModel  # noqa: E402
from dquartic.model.unet1d import UNet1d  # noqa: E402
from dquartic.utils.data_loader import DeviceBatchLoader, DIAMSDataset  # noqa: E402
from dquartic.utils.synthetic import synth_pool  # noqa: E402
from dquartic.utils.validation import ValidationSet, hold_out, validation_pairs  # noqa: E402

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


def kernel(reps=20, rounds=3):
    b = 64
    g = torch.Generator(device="cuda").manual_seed(0)
    truth = torch.rand(b, RT, MZ, device="cuda", generator=g) * (torch.rand(b, RT, MZ, device="cuda", generator=g) < 0.05)
    pred = truth + 0.01 * torch.randn(b, RT, MZ, device="cuda", generator=g)
    part = torch.empty(b * N.map_scores_nblk(MZ) * 9, dtype=torch.float64, device="cuda")
    out = torch.empty(b, 9, dtype=torch.float64, device="cuda")
    f = lambda: N.call("dq_map_scores", pred, truth, part, out, b, RT, MZ)
    f()
    torch.cuda.synchronize()
    best = float("inf")
    for _ in range(rounds):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            f()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) / reps)
    n = b * RT * MZ
    print(f"dq_map_scores {b} x {RT} x {MZ}: {best * 1e3:8.1f} us  {8 * n / (best * 1e-3) / 1e12:.2f} TB/s "
          f"(8 B/element, best of {rounds} rounds of {reps})", flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    print(card(), flush=True)
    kernel()

    torch.manual_seed(1234)
    net = UNet1d(dim=CFG["dim"], channels=1, dim_mults=CFG["dim_mults"], conditional=True, init_cond_channels=1,
                 attn_cond_channels=1, downsample_dim=CFG["downsample_dim"], simple=True, device="cuda")
    d = DDIMDiffusionModel(net, device="cuda")
    ms2, ms1 = synth_pool(520, RT, MZ, seed=1234)
    with tempfile.TemporaryDirectory() as tmp:
        np.save(os.path.join(tmp, "ms2.npy"), ms2)
        np.save(os.path.join(tmp, "ms1.npy"), ms1)
        del ms2, ms1
        full = DIAMSDataset(ms2_file=os.path.join(tmp, "ms2.npy"), ms1_file=os.path.join(tmp, "ms1.npy"),
                            normalize="minmax")
        split = DIAMSDataset(ms2_file=os.path.join(tmp, "ms2.npy"), ms1_file=os.path.join(tmp, "ms1.npy"),
                             normalize="minmax")
        lo, hi = hold_out(split, 0.1)
        pairs = validation_pairs(split, lo, hi, 64, seed=0)
        loaders = {"no validation": DeviceBatchLoader(full, 256, "cuda", pool="hbm", batches_per_epoch=3),
                   "10 % held out + validate": DeviceBatchLoader(split, 256, "cuda", pool="hbm", batches_per_epoch=3)}
    vset = ValidationSet(loaders["10 % held out + validate"], pairs, 1000, bands=10, seed=0)

    # 2. validate alone
    d.validate(vset)   # warm-up
    for _ in range(args.rounds):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        v = d.validate(vset)
        torch.cuda.synchronize()
        s = time.perf_counter() - t0
        print(f"validate 64 windows x 10 bands, chunk 64: {s:.3f} s = {640 / s:.0f} forwards/s  "
              f"(val_loss {v['val_loss']:.6f})", flush=True)

    # 3. training epochs with and without validation, alternated
    d._prepare_training(1e-5)
    random.seed(0)
    for name, loader in loaders.items():   # warm-up of both arms
        d._train_one_epoch(0, loader)
    times = {k: [] for k in loaders}
    for r in range(args.rounds):
        for name, loader in loaders.items():
            loader.dataset.reset_epoch()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            d._train_one_epoch(r, loader)
            if loader.dataset.n_train < len(loader.dataset):
                d.validate(vset)
            torch.cuda.synchronize()
            times[name].append(time.perf_counter() - t0)
    for name, ts in times.items():
        print(f"training epoch (3 steps of batch 256), {name:26s}: " + ", ".join(f"{t:.3f}" for t in ts)
              + f" s; median {np.median(ts):.3f} s", flush=True)
    diff = [b - a for a, b in zip(*times.values())]
    print("validation cost per epoch, round by round: " + ", ".join(f"{x:+.3f}" for x in diff) + " s", flush=True)

    # 4. dquartic evaluate's body with dpm++2m@20
    d.model.eval()
    for _ in range(2):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = cli.evaluate_model(d, vset, sampler="dpm++2m", num_steps=20, seed=0, chunk=32)
        torch.cuda.synchronize()
        s = time.perf_counter() - t0
        m = res["samplers"]["dpm++2m@20"]["mean"]
        print(f"evaluate_model (validate + dpm++2m@20 on 64 windows, chunk 32): {s:.2f} s; mean cosine "
              f"{m['cosine']:.4f}, rmse {m['rmse']:.4f}, spectral angle {m['spectral_angle']:.4f}, XIC corr "
              f"{m['xic_corr']:.4f} (untrained weights)", flush=True)


if __name__ == "__main__":
    main()
