"""bench.py — headline benchmark of the B200-native dquartic hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): default denoiser (1,204,738,391 parameters, dquartic_train_config.json),
bf16 tensor-core mid stage / fp32 elsewhere, synthetic multiplexed MS2 maps of the config's shape
(34 x 40000), batch 256 per GPU.  A "step" is one optimizer step over one batch: multiplexing of 256 drawn pairs,
q_sample, U-Net forward/backward (gradient accumulation over 4 micro-batches of 64), epsilon-MSE, grad-clip 10 + AdamW.
N > 1 (torchrun): weak scaling, 256 samples per GPU, one bucketed NCCL gradient all-reduce per step.

One JSON line on rank 0:
  value      train samples/s, inputs resident in HBM (slice pool of 520 in HBM; pair drawing, multiplexing / normalisation
             kernel, q_sample, forward / backward, clip + AdamW all inside the timed loop)
  e2e        the same through the public API with HOST buffers: pool in pinned host memory, per-step H2D copy of
             the drawn raw slices, loss read back to the host every step
  roofline   dominant kernel (measured live with CUDA events), see DESIGN.md
  cpu_baseline        the UNMODIFIED reference (vendored by oracle/make_ref.py into oracle/_ref) on the host cores, bounded
                      sample; the oracle port if oracle/_ref is absent
  gpu_eager_baseline  the same reference code on the B200 in eager fp32 ("stock PyTorch on B200", SURVEY.md §8d), b = 1 and
                      the largest batch <= 8 that fits
  sampling   DDIM-sampled MS2 maps/s (50 steps) through DDIMDiffusionModel.sample_windows, windows sharded over the ranks
  strong     (N > 1) the same step at a GLOBAL batch of 256 (256 / N per GPU); dp_check: N-rank gradient vs one rank on
             the union batch
`--impl reference` times the reference's own `_train_one_batch` (oracle/_ref) on the host cores, one sample per step.

`--dump-outputs DIR` writes what the last timed step of `value` handed its caller, as float32 / float64 .npy files, so
that two builds run with the same arguments (hence the same inputs) can be compared output for output (`bench_outputs/`
at the repository root is git-ignored):
  loss.npy               the mean loss `_train_one_batch` returned (float64 scalar)
  x0.npy, ms2_cond.npy   the multiplexed batch, 2^20 fixed, seeded positions of each
  ms1_cond.npy           the MS1 conditioning of the batch, whole
  params.npy, grads.npy  the parameters after the optimizer step and the step's gradients: per parameter tensor, in
                         state-dict order, all of it or 4096 fixed, seeded positions; the two arrays line up element
                         for element, with zeros in grads.npy for tensors without a gradient (the rotary freqs).
                         With N > 1 ranks they come from rank 0, and grads.npy is rank 0's gradient buffer after the
                         exchange: under the sharded optimizer only the pieces rank 0 owns hold the reduced sum
"""
import argparse
import atexit
import json
import os
import random
import shutil
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "diffusion-deconvolution-dia-msms-data_b200"))

DEFAULT_CFG = dict(dim=4, channels=1, dim_mults=[1, 2, 2, 3, 3, 4, 4], conditional=True, init_cond_channels=1,
                   attn_cond_channels=1, tfer_dim_mult=620, downsample_dim=40000, simple=True)
RT, MZ = 34, 40000
FWD_GFLOP_PER_SAMPLE = 212.87  # SURVEY.md §8d (FlopCounterMode on the reference at b = 1)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tensor=d["bf16_tflops"], tensor_sustained=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tensor=1590.0, tensor_sustained=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""

    def __init__(self, index=0):
        self.lines = []
        self.proc = None
        self.index = index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "200"], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------- reference arm
def _ref_path():
    p = os.path.join(ROOT, "oracle", "_ref")
    return p if os.path.isdir(os.path.join(p, "dquartic", "model")) else None


def ref_train_step_rate(torch, device, batch, steps, warmup):
    """The UNMODIFIED reference (oracle/_ref, vendored by oracle/make_ref.py): DDIMDiffusionModel._train_one_batch =
    zero_grad, train_step (q_sample, U-Net forward, MSE), backward, clip_grad_norm_(10), AdamW.step, loss.item() on
    `device`, full-size default model, fp32.  Returns (samples/s, description)."""
    rp = _ref_path()
    if rp not in sys.path:
        sys.path.insert(0, rp)
    import importlib
    mods = [m for m in list(sys.modules) if m == "dquartic" or m.startswith("dquartic.")]
    saved = {m: sys.modules.pop(m) for m in mods}      # our package has the same name: import the reference's, then restore
    try:
        unet = importlib.import_module("dquartic.model.unet1d")
        model = importlib.import_module("dquartic.model.model")
    finally:
        for m in list(sys.modules):
            if m == "dquartic" or m.startswith("dquartic."):
                sys.modules.pop(m)
        sys.modules.update(saved)
        sys.path.remove(rp)
    torch.manual_seed(0)
    net = unet.UNet1d(dim=DEFAULT_CFG["dim"], channels=1, dim_mults=tuple(DEFAULT_CFG["dim_mults"]), conditional=True,
                      init_cond_channels=1, attn_cond_channels=1, tfer_dim_mult=620, downsample_dim=MZ, simple=True).to(device)
    d = model.DDIMDiffusionModel(net, device=device)
    d._set_lr(1e-5)
    g = torch.Generator().manual_seed(0)
    x0 = (torch.rand(batch, RT, MZ, generator=g) * (torch.rand(batch, RT, MZ, generator=g) < 0.02)).to(device)
    other = (torch.rand(batch, RT, MZ, generator=g) * (torch.rand(batch, RT, MZ, generator=g) < 0.02)).to(device)
    cond = 0.5 * x0 + 0.5 * other
    ms1 = torch.rand(batch, RT, generator=g).to(device)
    times = []
    for it in range(warmup + steps):
        if device != "cpu":
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        d._train_one_batch(x0, ms2_cond=cond, ms1_cond=ms1)     # ends in loss.item(): a device sync
        if device != "cpu":
            torch.cuda.synchronize()
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    mean = sum(times) / len(times)
    del d, net
    return batch / mean, (f"{len(times)} optimizer step(s) at batch {batch} of the unmodified reference "
                          f"(_train_one_batch: fwd+bwd+clip+AdamW), full-size model, fp32, {mean:.3f} s/step")


def run_reference(args, rank, world, emit):
    """The reference's own CPU implementation of the training step, one sample per step, all host threads."""
    if rank != 0:
        return
    import torch

    cores = os.cpu_count()
    torch.set_num_threads(cores)
    if _ref_path():
        v, sample = ref_train_step_rate(torch, "cpu", 1, steps=args.steps, warmup=args.warmup)
        kind = "reference"
    else:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import dquartic_oracle as O
        v, sample = cpu_train_step_rate(O, torch, steps=args.steps, warmup=args.warmup)
        kind = "port"
    ms = 1000.0 / v
    line = {
        "impl": "reference", "metric": "train_samples_per_s", "value": v, "unit": "samples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(1, 1, per_gpu_batch=1),
        "cpu_baseline": {"value": v, "unit": "samples/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def cpu_train_step_rate(O, torch, steps, warmup):
    """fwd + bwd + clip + AdamW of ONE full-size sample per step on the CPU (batched oracle at b = 1)."""
    cfg = DEFAULT_CFG
    P = {}
    g = torch.Generator().manual_seed(0)
    for name, shape in O.param_shapes(cfg).items():
        if name.endswith("freqs"):
            P[name] = O.rotary_freqs()
            continue
        fan_in = 1
        for s in shape[1:]:
            fan_in *= s
        if name.endswith(".g"):
            P[name] = torch.ones(shape)
        else:
            P[name] = (torch.rand(shape, generator=g) * 2 - 1) / max(1.0, fan_in) ** 0.5
        P[name].requires_grad_(True)
    _, _, ab = O.schedule_tables(1000, "cosine")
    names = [k for k in P if P[k].requires_grad]
    m = {k: torch.zeros_like(P[k]) for k in names}
    v = {k: torch.zeros_like(P[k]) for k in names}
    x0 = torch.rand(1, RT, MZ, generator=g) * (torch.rand(1, RT, MZ, generator=g) < 0.02)
    other = torch.rand(1, RT, MZ, generator=g) * (torch.rand(1, RT, MZ, generator=g) < 0.02)
    cond = O.mix(x0, other)
    ms1 = torch.rand(1, RT, generator=g)
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        t = torch.randint(0, 1000, (1,), generator=g)
        noise = torch.randn(1, RT, MZ, generator=g)
        for k in names:
            P[k].grad = None
        loss, _ = O.train_loss(P, cfg, ab, x0, cond, ms1, t, noise)
        loss.backward()
        with torch.no_grad():
            grads, _ = O.clip_grad_norm([P[k].grad for k in names])
            for k, gk in zip(names, grads):
                p_new, m[k], v[k] = O.adamw_step(P[k], gk, m[k], v[k], it + 1, 1e-5)
                P[k].copy_(p_new)
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    mean = sum(times) / len(times)
    return 1.0 / mean, f"{len(times)} optimizer step(s) at batch 1 (fwd+bwd+clip+AdamW), full-size model, fp32, {mean:.1f} s/step"


def workload_config(world, micro_batch, per_gpu_batch):
    return {
        "workload": "configs[1]: default DDIM denoiser (1,204,738,391 params), synthetic multiplexed MS2 34x40000, "
                    f"batch {per_gpu_batch}/GPU, one optimizer step per bench step",
        "per_gpu_batch": per_gpu_batch, "global_batch": per_gpu_batch * world, "micro_batch": micro_batch,
        "rt": RT, "mz": MZ, "parallelism": f"dp{world}", "l2": "inputs larger than L2 (activations >> 126 MB per step)",
    }


DUMP_BATCH_ELEMS = 1 << 20
DUMP_PER_TENSOR = 4096


def _sample_positions(torch, np, rng, t, k):
    """Index tuple of k seeded positions of `t` (sorted, drawn with replacement), or of every position if it has <= k."""
    n = t.numel()
    flat = np.arange(n) if n <= k else np.sort(rng.integers(0, n, size=k))
    return tuple(torch.from_numpy(i).to(t.device) for i in np.unravel_index(flat, tuple(t.shape)))


def dump_outputs(out_dir, torch, np, net, last):
    """--dump-outputs: see the module docstring.  The positions come from one fixed seed and depend only on the shapes,
    so every build of the same model samples the same elements."""
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(1234)
    arrays = {"loss": np.float64(last["loss"])}
    for name in ("x0", "ms2_cond"):
        t = last[name]
        arrays[name] = t[_sample_positions(torch, np, rng, t, DUMP_BATCH_ELEMS)].float().cpu().numpy()
    arrays["ms1_cond"] = last["ms1_cond"].float().cpu().numpy()
    net.sync_params()
    ps, gs = [], []
    for _, p in net.named_parameters():
        idx = _sample_positions(torch, np, rng, p, DUMP_PER_TENSOR)
        ps.append(p.detach()[idx].float().cpu())
        gs.append(torch.zeros_like(ps[-1]) if p.grad is None else p.grad[idx].float().cpu())
    arrays["params"] = torch.cat(ps).numpy()
    arrays["grads"] = torch.cat(gs).numpy()
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------- our arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--batch", type=int, default=256, help="samples per GPU per optimizer step")
    ap.add_argument("--micro-batch", type=int, default=64)
    ap.add_argument("--pool", type=int, default=520, help="synthetic pool size (slices; 520 = the notebooks' pool, SURVEY.md §8d)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sampling", action="store_true")
    ap.add_argument("--sample-windows", type=int, default=1024, help="DDIM windows per GPU streamed through sample_windows")
    ap.add_argument("--sample-chunk", type=int, default=64)
    ap.add_argument("--no-eager-baseline", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as .npy files to DIR")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries the ONE JSON line only: libraries that write to file descriptor 1 (NCCL prints its version there,
    # the dataset prints an "Info: Loaded .." line as the reference does) are sent to stderr for the duration of the run
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())

    if args.impl == "reference":
        return run_reference(args, rank, world, emit)

    import numpy as np
    import torch
    import torch.distributed as dist

    from dquartic import _native as N
    from dquartic.model.model import DDIMDiffusionModel
    from dquartic.model.unet1d import UNet1d
    from dquartic.utils.data_loader import DeviceBatchLoader, DIAMSDataset
    from dquartic.utils.synthetic import synth_pool

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group(backend="nccl", device_id=dev)

    # ---- synthetic pool (same on every rank), written to npy so the public DIAMSDataset path is used
    import tempfile
    tmp = tempfile.mkdtemp(prefix=f"dq_bench_{rank}_")
    atexit.register(shutil.rmtree, tmp, ignore_errors=True)   # 2.8 GB at the default pool; the dataset maps it until exit
    ms2, ms1 = synth_pool(args.pool, RT, MZ, seed=1234)
    np.save(os.path.join(tmp, "ms2.npy"), ms2)
    np.save(os.path.join(tmp, "ms1.npy"), ms1)
    import contextlib
    with contextlib.redirect_stdout(sys.stderr):   # the dataset prints an "Info: Loaded .." line (as the reference does);
        ds = DIAMSDataset(ms2_file=os.path.join(tmp, "ms2.npy"), ms1_file=os.path.join(tmp, "ms1.npy"), normalize="minmax")
    # stdout carries the ONE JSON line only
    random.seed(1234 + rank)
    torch.manual_seed(1234 + rank)

    # ---- model (random init of the default architecture, identical on every rank)
    cfg = DEFAULT_CFG
    gen_state = torch.random.get_rng_state()
    torch.manual_seed(1234)
    net = UNet1d(dim=cfg["dim"], channels=1, dim_mults=tuple(cfg["dim_mults"]), conditional=True, init_cond_channels=1,
                 attn_cond_channels=1, downsample_dim=cfg["downsample_dim"], simple=True, device=dev)
    torch.random.set_rng_state(gen_state)
    if world > 1:
        dist.broadcast(net.flat_params(), src=0)
        net.mark_params_modified()
    ddim = DDIMDiffusionModel(net, device=dev)
    ddim.micro_batch = args.micro_batch
    ddim._prepare_training(1e-5)
    B = args.batch

    hbm_loader = DeviceBatchLoader(ds, B, dev, pool="hbm")
    pin_loader = DeviceBatchLoader(ds, B, dev, pool="pinned")


    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def draw(loader):
        ds.reset_epoch()
        return loader.draw(B)

    # ---- value: inputs resident in HBM when the timed region starts
    last = {}   # --dump-outputs: what the last timed step of `value` handed its caller

    def run_loop(n_warm, n_timed, e2e, keep_last=False):
        loader = pin_loader if e2e else hbm_loader
        for i in range(n_warm):
            if e2e:
                x0, m1, other, m2 = loader.make_batch(draw(loader))
                x0, m1c, cond = ddim._mix_to_device(x0, m1, other, (0.5, 0.5))
                ddim._train_one_batch(x0, cond, m1c)
            else:
                x0, m1, other, m2, cond = loader.make_batch(draw(loader), want_cond=True)
                ddim._train_one_batch(x0, cond, m1)
        barrier()
        l0 = N.launches
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        if e2e:
            nxt = draw(loader)
            loader.prefetch(nxt)
        for i in range(n_timed):
            if e2e:
                # public loader path: the distinct raw slices of THIS step's batch are copied host -> device from the
                # pinned pool inside the timed region (side stream), overlapped with the previous step's kernels
                pairs = nxt
                x0, m1, other, m2 = loader.make_batch(pairs)
                if i + 1 < n_timed:
                    nxt = draw(loader)
                    loader.prefetch(nxt)
                x0, m1c, cond = ddim._mix_to_device(x0, m1, other, (0.5, 0.5))
                ddim._train_one_batch(x0, cond, m1c)  # returns loss.item(): device -> host read every step
            else:
                # pool resident in HBM: pair drawing (host, python `random` as in the reference), then ONE kernel chain
                # gathers / normalises / mixes the 256 drawn pairs; all inside the timed region
                x0, m1, other, m2, cond = loader.make_batch(draw(loader), want_cond=True)
                loss = ddim._train_one_batch(x0, cond, m1)
        ev1.record()
        barrier()
        if keep_last:
            last.update(loss=loss, x0=x0, ms2_cond=cond, ms1_cond=m1)
        ms = ev0.elapsed_time(ev1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms, N.launches - l0

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_total, launches = run_loop(args.warmup, args.steps, e2e=False, keep_last=bool(args.dump_outputs))
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, torch, np, net, last)
    last.clear()
    ms_step = ms_total / args.steps
    value = B * world / (ms_step / 1000.0)

    ms_e2e_total, _ = run_loop(1, args.steps, e2e=True)
    ms_e2e = ms_e2e_total / args.steps
    e2e_value = B * world / (ms_e2e / 1000.0)
    h2d = pin_loader.h2d_bytes
    d2h = 4

    extra = {}
    if world > 1 and not args.no_strong:
        # strong scaling: the SAME global batch of 256 spread over the ranks (SURVEY.md §8d asks for both)
        Bw, mbw = B, ddim.micro_batch
        B = max(1, Bw // world)
        ddim.micro_batch = min(mbw, B)
        hbm_loader.batch_size = B
        ms_s, _ = run_loop(2, args.steps, e2e=False)
        strong = {"global_batch": B * world, "per_gpu_batch": B, "ms_per_step": ms_s / args.steps,
                  "value": B * world / (ms_s / args.steps / 1000.0), "unit": "samples/s", "scaling": "strong",
                  "note": "efficiency = value / (the N = 1 line's value): computed by the reader, not here"}
        B, ddim.micro_batch = Bw, mbw
        hbm_loader.batch_size = B
        dp = dp_check(torch, dist, ddim, net, dev, rank, world)
        if rank == 0:
            extra["strong"] = strong
            extra["dp_check"] = dp
    if rank == 0:
        extra["roofline"] = dominant_kernel_roofline(torch, N, net, dev, min(B, args.micro_batch))
        extra["step_breakdown"] = {"train_gflop_per_sample": 3 * FWD_GFLOP_PER_SAMPLE,
                                   "achieved_tflops_whole_step": 3 * FWD_GFLOP_PER_SAMPLE * B / ms_step,
                                   "frac_of_bf16_sustained_peak": 3 * FWD_GFLOP_PER_SAMPLE * B / ms_step / peaks()["tensor_sustained"]}
    if not args.no_sampling:
        extra_s = sampling_rate(torch, dist, ddim, hbm_loader, ds, dev, rank, world, args.sample_windows, args.sample_chunk)
        if rank == 0:
            extra["sampling"] = extra_s
    tc_err = N.la_tc_last_error()
    if tc_err is not None:
        raise RuntimeError(f"tcgen05 LinearAttention pipeline timed out during the bench: {tc_err}")
    if rank == 0 and world == 1 and not args.no_eager_baseline and _ref_path():
        # "stock PyTorch on B200": the unmodified reference in eager fp32 on the same GPU.  Our model and optimizer
        # state are released first (the eager reference materialises ~35 GB of activations per sample).
        hbm_loader.ms2 = pin_loader.ms2 = None
        del ddim, net
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        eager = []
        for bb in (1, 2, 4, 8):
            try:
                v, sample = ref_train_step_rate(torch, "cuda", bb, steps=2, warmup=1)
                eager.append({"batch": bb, "value": v, "unit": "samples/s", "sample": sample})
            except torch.cuda.OutOfMemoryError:
                eager.append({"batch": bb, "value": None, "note": "out of memory (180 GB) in eager fp32"})
                break
            except RuntimeError as e:   # the reference only runs at batch 1 (SURVEY.md finding 1)
                eager.append({"batch": bb, "value": None, "note": "the reference raises: " + str(e).splitlines()[0][:160]})
                break
            finally:
                gc.collect()
                torch.cuda.empty_cache()
        extra["gpu_eager_baseline"] = {"kind": "reference", "dtype": "f32", "device": torch.cuda.get_device_name(dev),
                                       "runs": eager,
                                       "note": "the reference only runs at batch 1 (SURVEY.md finding 1: its conditioning "
                                               "concat breaks for b > 1); the attempt at b = 2 is recorded as it fails"}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count()
        torch.set_num_threads(cores)
        if _ref_path():
            v, sample = ref_train_step_rate(torch, "cpu", 1, steps=1, warmup=0)
            kind = "reference"
        else:
            sys.path.insert(0, os.path.join(ROOT, "oracle"))
            import dquartic_oracle as O
            v, sample = cpu_train_step_rate(O, torch, steps=1, warmup=0)
            kind = "port"
        extra["cpu_baseline"] = {"value": v, "unit": "samples/s", "cores": cores, "kind": kind, "sample": sample}

    if rank == 0:
        line = {
            "metric": "train_samples_per_s", "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16 (mid-stage tcgen05 GEMMs, fp32 accumulate) / tf32 (linear-attention and 8-16-channel conv-backward mma.sync, fp32 accumulate) / f32 elsewhere",
            "data": "synthetic", "config": workload_config(world, args.micro_batch, B),
            "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e},
            "gpu_launches": int(launches), "clocks": clocks,
        }
        line.update(extra)
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def _time_ms(torch, fn, reps=3, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(reps):
        fn()
    ev1.record()
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1) / reps


def dominant_kernel_roofline(torch, N, net, dev, n_samples=64):
    """Live CUDA-event timings (torch's current stream = the launch stream) of the kernel families of the step at the
    shapes of one micro-batch (n_samples).  `roofline` = the family with the largest share of the step
    (profiles/): the LinearAttention backward at level 0 (C = 4, L = 40000).  Algorithmic work (DESIGN.md §4):
    the reference's four backward bmm's = 2 x 557056 x L FLOP per sample and level (SURVEY.md §3.3/§8d)."""
    pk = peaks()
    R, C, L = n_samples * RT, 4, MZ
    net._ensure_grads()
    others = []
    # ---- LinearAttention, level 0
    pre = "downs.0.2"
    x = torch.randn(R, C, L, device=dev)
    dres = torch.randn(R, C, L, device=dev)
    out, saved = net._la_fwd(pre, x, True)
    ms_f = _time_ms(torch, lambda: net._la_fwd(pre, x, True))
    ms_b = _time_ms(torch, lambda: net._la_bwd(pre, saved, dres))
    fl_f = 557056.0 * L * n_samples
    ach_b = 2.0 * fl_f / (ms_b * 1e-3) / 1e12
    # exp count: 128 (k) + 128 (q) per position forward, recomputed in backward; MUFU.EX2 = 16 / clk / SM
    exp_floor_ms = lambda n_exp: n_exp * R * L / (148 * 16 * 1.965e9) * 1e3
    main = {"kernel": f"dq_linattn_bwd (la_bwd_q_tc [tcgen05 / TMEM] + la_bwd_combine + la_bwd_kv [mma.sync]), level 0 (C=4, L=40000), {n_samples} samples",
            "bound": "tensor", "achieved": ach_b, "peak": pk["tensor"], "unit": "TFLOP/s", "frac": ach_b / pk["tensor"],
            # dram__bytes_read.sum + dram__bytes_write.sum of la_bwd_q + la_bwd_combine + la_bwd_kv at exactly this shape
            # (C = 4, L = 40000, 64 samples), one `ncu --set full` capture: profiles/r2c_la_bwd64_ncu_full_summary.txt
            # (5.603 + 0.056 + 5.576 GB; the round-1 kernels moved the same bytes)
            "traffic": (11.235e9 if n_samples == 64 else None), "traffic_unit": "bytes per dq_linattn_bwd call",
            "ms_per_launch": ms_b, "peak_source": pk["src"],
            "note": "algorithmic FLOPs = the reference's 32x32 per-head bmm's; the kernels factor them through the C "
                    "input channels (32xC products, ~1/4 of the MMA work at C=4; q path: tcgen05.mma kind::tf32 / f16 with TMEM "
                    "score rings, k/v path: mma.sync TF32) and are bound by MUFU.EX2 + instruction issue + the small-MMA "
                    "pipeline skeleton (DESIGN.md section 4), not by the tensor pipe or HBM: MUFU floor "
                    f"{exp_floor_ms(256):.2f} ms vs {ms_b:.2f} ms measured; HBM-algorithmic bytes "
                    f"{8 * C * 4 * R * L / 1e9:.2f} GB = {8 * C * 4 * R * L / 1e9 / (ms_b * 1e-3):.0f} GB/s"}
    others.append({"kernel": f"dq_linattn_fwd (la_stats + la_combine + la_out), level 0, {n_samples} samples", "bound": "tensor",
                   "achieved": fl_f / (ms_f * 1e-3) / 1e12, "peak": pk["tensor"], "unit": "TFLOP/s",
                   "frac": fl_f / (ms_f * 1e-3) / 1e12 / pk["tensor"], "ms_per_launch": ms_f,
                   "note": f"MUFU floor {exp_floor_ms(256):.2f} ms"})
    del x, dres, out, saved
    # ---- fused conv Block forward / backward, level 0 (C = 4 -> 4): HBM-bound
    b = n_samples
    net._time_path_fwd(torch.zeros(b, dtype=torch.long, device=dev), b, False)
    net._dSS = torch.zeros(b, net.ss_total, device=dev)
    pre = "downs.0.0"
    w, bn, gname, sso = pre + ".block1.proj.weight", pre + ".block1.proj.bias", pre + ".block1.norm.g", net.ss_off[pre + ".mlp.1"]
    x1 = torch.randn(R, C, L, device=dev)
    y, u = net._conv_fwd(x1, None, w, bn, 3, 1, 1, 1, L, g=gname, ss=sso, act=1, save_u=True, rps=RT)
    dy = torch.randn_like(y)
    ms = _time_ms(torch, lambda: net._conv_fwd(x1, None, w, bn, 3, 1, 1, 1, L, g=gname, ss=sso, act=1, save_u=True, rps=RT))
    by = 3 * C * 4.0 * R * L   # read x, write u and y
    others.append({"kernel": "dq_conv1d_fwd (conv_fwd_tma_kernel<4,3>: conv k3 + RMSNorm + scale/shift + SiLU), level 0",
                   "bound": "hbm", "achieved": by / (ms * 1e-3) / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                   "frac": by / (ms * 1e-3) / 1e9 / pk["hbm"], "ms_per_launch": ms})
    ms = _time_ms(torch, lambda: net._conv_bwd_fused(dy, u, gname, sso, 1, x1, None, w, bn, 3, rps=RT))
    by = 4 * C * 4.0 * R * L   # read dy, u, x, write dx
    others.append({"kernel": "dq_conv_bwd_fused (conv_bwd_fused_tma_kernel<4,3>: epilogue bwd + dgrad + wgrad), level 0",
                   "bound": "hbm", "achieved": by / (ms * 1e-3) / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                   "frac": by / (ms * 1e-3) / 1e9 / pk["hbm"], "ms_per_launch": ms})
    del x1, y, u, dy
    # ---- ResnetBlock backward on the up path at 8 channels (ups.4.0: 16 -> 8, L = 10000): block2, then block1 fused with
    # the 1x1 res_conv; dgrad / wgrad contractions on mma.sync TF32 tensor cores inside the HBM pipeline
    pre, c1, c2, L8 = "ups.4.0", 8, 8, 10000
    xa = torch.randn(R, c1, L8, device=dev)
    xb = torch.randn(R, c2, L8, device=dev)
    o8, saved8 = net._resnet_fwd(pre, xa, xb, RT, True)
    d8 = torch.randn_like(o8)
    ms = _time_ms(torch, lambda: net._resnet_bwd(pre, saved8, d8, RT))
    by = (7 * 8 + 2 * 16) * 4.0 * R * L8   # dout, u2, h1 -> dh1 | dh1, u1, x, dout -> dx
    others.append({"kernel": "ResnetBlock backward ups.4.0 (2 x conv_bwd_fused_tma_kernel<8,3>, TF32 mma.sync contractions, "
                             "res_conv fused), L = 10000", "bound": "hbm", "achieved": by / (ms * 1e-3) / 1e9,
                   "peak": pk["hbm"], "unit": "GB/s", "frac": by / (ms * 1e-3) / 1e9 / pk["hbm"], "ms_per_launch": ms})
    net._dSS = None
    del xa, xb, o8, saved8, d8
    # ---- mid-stage tcgen05 GEMMs (M = 32 x 36 padded rows, N = 10000, K = 3 x 10000)
    Nm, Mp = net.mid_channels, n_samples * (RT + 2)
    A = torch.randn(Mp, Nm, device=dev).bfloat16()
    W = torch.randn(3, Nm, Nm, device=dev).bfloat16()
    U = torch.empty(Mp, Nm, device=dev)
    ms = _time_ms(torch, lambda: net._gemm(A, Mp, Nm, Nm, W, Nm, Nm, Nm, Nm * Nm, 3, U, Nm, None, 0, Mp, Nm, Nm, 3,
                                           (-1, 0, 1), (0, 0, 0), (0, 0, 0), (0, 1, 2)), reps=5)
    fl = 2.0 * Mp * Nm * Nm * 3
    others.append({"kernel": f"dq_gemm_bf16_tn (tcgen05 3-tap implicit GEMM, mid Conv1d(10000,10000,3) fwd/dgrad), M={Mp}",
                   "bound": "tensor", "achieved": fl / (ms * 1e-3) / 1e12, "peak": pk["tensor"], "unit": "TFLOP/s",
                   "frac": fl / (ms * 1e-3) / 1e12 / pk["tensor"], "ms_per_launch": ms})
    Kc = 256 * (RT + 2)   # weight gradient of one optimizer step: all micro-batches of the 256-sample batch along K
    dUT = torch.randn(Nm, Kc, device=dev).bfloat16()
    AT3 = torch.randn(3, Nm, Kc, device=dev).bfloat16()
    dW = torch.zeros(3, Nm, Nm, device=dev)
    ms = _time_ms(torch, lambda: net._gemm(dUT, Nm, Kc, Kc, AT3, Nm, Kc, Kc, Nm * Kc, 3, dW, Nm, None, 1, Nm, Nm, Kc, 1,
                                           (0,), (0,), (0,), (0,), nz=3, z_b_tap_step=1, z_c_stride=Nm * Nm), reps=2, warm=1)
    fl = 2.0 * Kc * Nm * Nm * 3
    others.append({"kernel": f"dq_gemm_bf16_tn (mid conv wgrad, K = {Kc} = 256 samples x 36 padded rows, fp32 accumulate into dW)",
                   "bound": "tensor", "achieved": fl / (ms * 1e-3) / 1e12, "peak": pk["tensor"], "unit": "TFLOP/s",
                   "frac": fl / (ms * 1e-3) / 1e12 / pk["tensor"], "ms_per_launch": ms})
    del A, W, U, dUT, AT3, dW
    net._gflat.zero_()
    main["others"] = others
    return main


def sampling_rate(torch, dist, ddim, loader, ds, dev, rank, world, windows, chunk):
    """BASELINE configs[3]: DDIM sampling (50 steps) of `windows` DIA windows PER GPU through the product driver
    `DDIMDiffusionModel.sample_windows`: windows sharded over the ranks in contiguous blocks, x_T from (seed, window id),
    the 50-step loop of a chunk replayed from one CUDA graph, results copied to pinned host memory, no collective.  The
    conditioning of window w is the multiplexed pair (w mod 64) of the synthetic pool (the pool is reused cyclically)."""
    ds.reset_epoch()
    x0p, m1p, otherp, m2p, condp = loader.make_batch(loader.draw(64), want_cond=True)
    del x0p, otherp, m2p

    def cond_fn(ids):
        idx = torch.tensor([w % 64 for w in ids], device=dev)
        return condp[idx], m1p[idx]

    total = windows * world
    ids = list(range(total))
    ddim.sample_windows(ids[: 2 * chunk * world], cond_fn, seed=1234, num_steps=2, chunk=chunk, rank=rank, world=world)  # warm-up
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    # the pinned result buffer of this rank is allocated before the timed region (a one-time host allocation of 5.4 MB per
    # window); everything else of the driver - x_T generation, graph capture of the first chunk, device -> host copies - is inside
    lo, hi = ddim.shard_windows(total, rank, world)
    out = torch.empty((hi - lo, RT, MZ), dtype=torch.float32).pin_memory()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    got, maps = ddim.sample_windows(ids, cond_fn, seed=1234, num_steps=50, chunk=chunk, rank=rank, world=world, out=out)
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t)
    ddim.model.train()
    v = total / (ms / 1000.0)
    tf = v * 50 * FWD_GFLOP_PER_SAMPLE / 1e3 / world   # TFLOP/s per GPU of reference-algorithmic forward work
    return {"metric": "ddim_maps_per_s", "value": v, "unit": "maps/s", "num_steps": 50, "windows_per_gpu": windows,
            "windows_total": total, "chunk": chunk, "ms_total": ms, "d2h_bytes": int(maps.numel() * 4),
            "forward_tflops_per_gpu": tf, "frac_of_bf16_sustained_peak": tf / peaks()["tensor_sustained"],
            "note": "forward = 212.87 GFLOP per map and step (SURVEY.md §8d); includes x_T generation, the device -> "
                    "pinned-host copy of every map and the CUDA-graph capture of the first chunk (the pinned result buffer "
                    "is allocated beforehand)"}


def dp_check(torch, dist, ddim, net, dev, rank, world, per_rank=2):
    """N-rank data-parallel step vs ONE rank on the union batch (same injected t / noise): cosine of the whole flat
    gradient (mean over the union batch).  lr = 0, so parameters stay put.  Runs on every rank; rank 0 reports."""
    import copy
    g = torch.Generator().manual_seed(4321)
    n = per_rank * world
    x0 = (torch.rand(n, RT, MZ, generator=g) * (torch.rand(n, RT, MZ, generator=g) < 0.02)).to(dev)
    cond = (0.5 * x0 + 0.5 * (torch.rand(n, RT, MZ, generator=g) * (torch.rand(n, RT, MZ, generator=g) < 0.02)).to(dev))
    m1 = torch.rand(n, RT, generator=g).to(dev)
    noise = torch.rand(n, RT, MZ, generator=g).to(dev)       # the harness maps injected noise n -> 2 n - 1
    t = torch.randint(0, 1000, (n,), generator=g).to(dev)
    lr = ddim.optimizer.param_groups[0]["lr"]
    ddim.optimizer.param_groups[0]["lr"] = 0.0
    ddim.optimizer.param_groups[0]["weight_decay"] = 0.0
    mb = ddim.micro_batch
    ddim.micro_batch = per_rank
    sl = slice(rank * per_rank, (rank + 1) * per_rank)
    ddim._train_one_batch(x0[sl], cond[sl], m1[sl], noise=noise[sl], t=t[sl])
    gsum = net.flat_grads()[: net.n_trainable_flat].clone()
    plan = ddim._shard_plan()
    if plan:                      # sharded exchange: every rank holds the reduced values of its pieces only
        for (o, cnt) in plan:
            k = cnt // world
            dist.all_gather_into_tensor(gsum[o:o + cnt], gsum[o + rank * k:o + (rank + 1) * k].clone())
    g_dp = gsum / world
    norm_dp = float(ddim.optimizer.last_grad_norm)
    # one rank, union batch, no exchange
    dist_on = ddim._dist_on
    ddim._dist_on = lambda: False
    real_allreduce = ddim._allreduce_grads
    ddim._allreduce_grads = lambda: 1.0
    real_step = ddim.optimizer.step
    ddim.optimizer.step = lambda *a, **k: None      # (the sharded optimizer's step is a collective; lr is 0 anyway)
    res = None
    if rank == 0:
        ddim._train_one_batch(x0, cond, m1, noise=noise, t=t)    # micro-batches of per_rank, accumulated
        g_ref = net.flat_grads()[: net.n_trainable_flat]
        num = float(torch.dot(g_dp.double(), g_ref.double()))
        cos = num / float(g_dp.double().norm() * g_ref.double().norm())
        res = {"ranks": world, "union_batch": n, "flat_gradient_cosine": cos,
               "max_abs_diff_over_max_abs": float((g_dp - g_ref).abs().max() / g_ref.abs().max()),
               "sharded_optimizer": bool(plan), "grad_norm_dp": norm_dp}
    ddim._dist_on = dist_on
    ddim._allreduce_grads = real_allreduce
    ddim.optimizer.step = real_step
    ddim.optimizer.param_groups[0]["lr"] = lr
    ddim.optimizer.param_groups[0]["weight_decay"] = 0.01
    ddim.micro_batch = mb
    dist.barrier()
    return res


if __name__ == "__main__":
    main()
