"""Speed of the few-step ODE samplers on one GPU, on the default denoiser (34 x 40000 maps).

1. maps/s through DDIMDiffusionModel.sample_windows (1024 windows, chunk 64: one CUDA graph per call, results copied
   to pinned host memory) for reference@50, ddim@20, dpm++2m@20 and dpm++2m@10; host clock around the call, which ends
   in a device synchronise.  Weights: the network's seeded initialisation (speed does not depend on them).  The
   conditioning of window w is pool window w mod 64 of a random pool on the device.
2. CUDA-event times of dq_dpm_step (first and second order) and dq_ddim_step at 64 x 34 x 40000 elements, the three
   alternated; bytes/s from 20 / 16 / 12 B per element.  The 1.0-1.7 GB per launch exceed the L2, so they stream
   from HBM.
3. The one-off cost a `dquartic predict` slice pays for its CUDA graph: sample_windows' 2-step warm-up plus the capture
   of the 20-step dpm++2m loop of one 64-window chunk, host clock with device synchronises.
4. `dquartic predict`'s body, `cli.predict_to_file`, on 256 int32 windows held in host memory (one slice of 4 chunks),
   dpm++2m@20, writing a .npy in a temporary directory, against sample_windows alone on the same windows: the
   difference is the per-window min-max scaling, the graph set-up, the de-normalisation and the file write.

Prints the card name and power limit first.  Usage: python tools/sampler_time.py [--windows W] [--chunk C]"""
import argparse
import os
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


def kernels(reps=20, rounds=3):
    n = 64 * RT * MZ
    x, out, hist = (torch.randn(n, device="cuda") for _ in range(3))
    xn = torch.empty_like(x)
    runs = {
        "dq_dpm_step 2nd order": (20, lambda: N.call("dq_dpm_step", x, out, hist, xn, None, 0.5, 0.8, 0, 0.9, 0.2,
                                                     1.3, -0.3, 0, n)),
        "dq_dpm_step 1st order": (16, lambda: N.call("dq_dpm_step", x, out, hist, xn, None, 0.5, 0.8, 0, 0.9, 0.2,
                                                     1.0, 0.0, 0, n)),
        "dq_ddim_step": (12, lambda: N.call("dq_ddim_step", x, out, xn, 0.5, 0.8, 0.6, 0.7, 0, n)),
    }
    for _, f in runs.values():
        f()
    torch.cuda.synchronize()
    best = {k: float("inf") for k in runs}
    for _ in range(rounds):
        for k, (_, f) in runs.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                f()
            e1.record()
            torch.cuda.synchronize()
            best[k] = min(best[k], e0.elapsed_time(e1) / reps)
    for k, (b, _) in runs.items():
        print(f"{k:24s} n={n}: {best[k] * 1e3:8.1f} us  {b * n / (best[k] * 1e-3) / 1e12:.2f} TB/s "
              f"({b} B/element, best of {rounds} rounds of {reps})")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=1024)
    ap.add_argument("--chunk", type=int, default=64)
    args = ap.parse_args()
    print(card())
    kernels()

    torch.manual_seed(1234)
    net = UNet1d(dim=CFG["dim"], channels=1, dim_mults=CFG["dim_mults"], conditional=True, init_cond_channels=1,
                 attn_cond_channels=1, downsample_dim=CFG["downsample_dim"], simple=True, device="cuda")
    d = DDIMDiffusionModel(net, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(0)
    pool2 = torch.rand(64, RT, MZ, device="cuda", generator=g) * (torch.rand(64, RT, MZ, device="cuda", generator=g) < 0.05)
    pool1 = torch.rand(64, RT, device="cuda", generator=g)

    def cond_fn(ids):
        idx = torch.tensor([w % 64 for w in ids], device="cuda")
        return pool2[idx], pool1[idx]

    ids = list(range(args.windows))
    out = torch.empty((args.windows, RT, MZ), dtype=torch.float32).pin_memory()
    d.sample_windows(ids[:2 * args.chunk], cond_fn, num_steps=2, chunk=args.chunk, rank=0, world=1)   # warm-up
    torch.cuda.synchronize()
    for sampler, steps in (("reference", 50), ("ddim", 20), ("dpm++2m", 20), ("dpm++2m", 10)):
        t0 = time.perf_counter()
        d.sample_windows(ids, cond_fn, seed=1234, num_steps=steps, chunk=args.chunk, rank=0, world=1, out=out,
                         sampler=sampler)
        torch.cuda.synchronize()
        s = time.perf_counter() - t0
        print(f"sample_windows {sampler:9s} @{steps:2d} steps: {args.windows} windows in {s:7.2f} s = "
              f"{args.windows / s:6.1f} maps/s  ({s / args.windows / steps * 1e3:.2f} ms per map and step)")

    # one predict slice's graph set-up, as sample_windows does it
    xT = torch.randn(args.chunk, RT, MZ, device="cuda")
    c2, c1 = cond_fn(ids[:args.chunk])
    with torch.no_grad():
        for _ in range(2):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            d.sample(xT.clone(), c2, c1, num_steps=2, sampler="dpm++2m")
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                d.sample(xT, c2, c1, num_steps=20, sampler="dpm++2m")
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            graph.replay()
            torch.cuda.synchronize()
            t3 = time.perf_counter()
            del graph
            print(f"graph set-up per predict slice (chunk {args.chunk}, dpm++2m@20): warm-up {1e3 * (t1 - t0):.0f} ms "
                  f"+ capture {1e3 * (t2 - t1):.0f} ms; one replay {1e3 * (t3 - t2):.0f} ms")

    n = 4 * args.chunk
    rng = np.random.default_rng(0)
    ms2 = (rng.random((n, RT, MZ), dtype=np.float32) * 4000 * (rng.random((n, RT, MZ), dtype=np.float32) < 0.05)
           ).astype(np.int32)
    ms1 = (rng.random((n, RT)) * 7e5).astype(np.int32)
    with tempfile.TemporaryDirectory() as tmp:
        for _ in range(2):
            t0 = time.perf_counter()
            d.sample_windows(ids[:n], cond_fn, seed=1234, num_steps=20, chunk=args.chunk, rank=0, world=1,
                             out=out[:n], sampler="dpm++2m")
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            cli.predict_to_file(d, ms2, ms1, os.path.join(tmp, "pred.npy"), sampler="dpm++2m", num_steps=20,
                                chunk=args.chunk)
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            print(f"{n} windows, dpm++2m@20: sample_windows {t1 - t0:.2f} s = {n / (t1 - t0):.1f} maps/s; "
                  f"predict_to_file (scale, sample, de-normalise, write .npy) {t2 - t1:.2f} s = {n / (t2 - t1):.1f} maps/s")


if __name__ == "__main__":
    main()
