"""`dquartic` command line — same commands and options as the reference (/root/reference/dquartic/cli.py:26-188):
`dquartic train CONFIG [--parquet_directory --ms2-data-path --ms1-data-path --batch-size --checkpoint-path
--use-wandb --threads]`, `dquartic generate-config`.  `--ema-decay` (model.ema_decay in the config) keeps an exponential
moving average of the weights in the checkpoints.  `--validation-fraction` (the optional config section "validation")
holds out slices and selects the best checkpoint by a held-out denoising loss.  `dquartic predict` (not in the
reference) deconvolves a run of windows with a checkpoint; `dquartic evaluate` scores a checkpoint on the held-out
mixtures.  Differences: `--batch-size/--threads` are cast to int (the
reference passes strings to DataLoader and fails, SURVEY.md §5); under torchrun (RANK/WORLD_SIZE in the
environment) each rank binds one GPU, joins an NCCL process group and trains a batch shard;
`generate-train-data` (offline ETL) is out of scope.
"""
import ast
import os

import click
import numpy as np
import torch

from .model.model import SAMPLERS, DDIMDiffusionModel
from .model.unet1d import UNet1d
from .utils.config_loader import generate_train_config, load_train_config
from .utils.data_loader import DeviceBatchLoader, DIAMSDataset
from .utils.validation import ValidationSet, check_section, hold_out, validation_pairs


class PythonLiteralOption(click.Option):
    def type_cast_value(self, ctx, value):
        if not isinstance(value, str):
            return value
        try:
            return ast.literal_eval(value)
        except Exception:
            raise click.BadParameter(value)


@click.group(chain=True)
@click.version_option(version="0.1.0+b200")
def cli():
    """
    Diffusion Deconvolution of DIA-MS/MS Data (D^4) - B200 build
    """


def _init_distributed():
    ws = int(os.environ.get("WORLD_SIZE", "1"))
    if ws <= 1:
        return 0, 1, 0
    rank = int(os.environ["RANK"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    torch.distributed.init_process_group(backend="nccl" if torch.cuda.is_available() else "gloo")
    return rank, ws, local


def _unet_from_config(config):
    if config["model"]["use_model"] == "UNet1d":
        u = config["model"]["UNet1d"]
        return UNet1d(dim=u["dim"], channels=u["channels"], dim_mults=tuple(u["dim_mults"]),
                      conditional=u["conditional"], init_cond_channels=u["init_cond_channels"],
                      attn_cond_channels=u["attn_cond_channels"], tfer_dim_mult=u["tfer_dim_mult"],
                      downsample_dim=u["downsample_dim"], simple=u["simple"])
    if config["model"]["use_model"] == "CustomTransformer":
        raise NotImplementedError("CustomTransformer is dead code under the reference's DDIM API (SURVEY.md finding 2)")
    raise ValueError(f"Invalid model class: {config['model']['use_model']}")


@cli.command()
@click.argument("config-path", type=click.Path(exists=True), required=True)
@click.option("--parquet_directory", default=None, help="Directory of Parquet slices. Mutually exclusive with the NPY paths. Overrides config file")
@click.option("--ms2-data-path", default=None, help="Path to MS2 data, overrides config file")
@click.option("--ms1-data-path", default=None, help="Path to MS1 data, overrides config file")
@click.option("--batch-size", default=None, help="Batch size for training, overrides config file")
@click.option("--checkpoint-path", default=None, help="Path to save the best model, overrides config file")
@click.option("--use-wandb", default=None, cls=PythonLiteralOption, help="Use wandb for logging, overrides config file")
@click.option("--threads", default=None, help="Number of threads for data loading, overrides config file")
@click.option("--ema-decay", default=None, type=click.FloatRange(0.0, 1.0, min_open=True, max_open=True),
              help="Keep an exponential moving average of the weights with this decay (e.g. 0.9999) and save it in the "
                   "checkpoints as ema_state_dict, overrides config file")
@click.option("--validation-fraction", default=None, type=float,
              help="Hold out this fraction of the slices (0 < f < 1, the last ones in file order) and select the best "
                   "checkpoint by their denoising loss, overrides validation.fraction of the config file")
def train(config_path, parquet_directory, ms2_data_path, ms1_data_path, batch_size, checkpoint_path, use_wandb, threads,
          ema_decay, validation_fraction):
    """
    Train a DDIM model on the DIAMS dataset.
    """
    rank, world, local = _init_distributed()
    if rank == 0:
        click.echo("--" * 30)
        if torch.cuda.is_available():
            click.echo("GPU Information:")
            for i in range(torch.cuda.device_count()):
                print(f"GPU {i}: {torch.cuda.get_device_name(i)}")
                print(f"Total Memory: {torch.cuda.get_device_properties(i).total_memory / (1024 ** 2)} MB")
        else:
            print("No GPUs available.")
        click.echo("--" * 30)
        click.echo(f"Info: Loading config from {config_path}")

    config = load_train_config(config_path, parquet_directory=parquet_directory, ms2_data_path=ms2_data_path,
                               ms1_data_path=ms1_data_path, batch_size=batch_size, checkpoint_path=checkpoint_path,
                               use_wandb=use_wandb, threads=threads, ema_decay=ema_decay,
                               validation_fraction=validation_fraction)
    val_cfg = _validation_section(config, for_train=True)
    batch_size = int(config["model"]["batch_size"])
    checkpoint_path = config["model"]["checkpoint_path"]
    use_wandb = config["wandb"]["use_wandb"]

    if not torch.cuda.is_available():
        raise RuntimeError("the B200 build of dquartic has no CPU training path")
    device = torch.device("cuda", local)
    dataset = DIAMSDataset(config["data"]["parquet_directory"], config["data"]["ms2_data_path"],
                           config["data"]["ms1_data_path"], normalize=config["data"]["normalize"])
    if val_cfg is not None:
        val_pairs = _validation_pairs(dataset, val_cfg)
    if world > 1:
        import random
        random.seed(1234 + rank)  # each rank draws its own pairs, like DataLoader workers do in the reference
    per_rank = max(1, batch_size // world)
    data_loader = DeviceBatchLoader(dataset, per_rank, device, pool="hbm",
                                    batches_per_epoch=(dataset.n_train + batch_size - 1) // batch_size)

    model = _unet_from_config(config).to(device)
    if world > 1:  # identical initial weights on every rank
        torch.distributed.broadcast(model.flat_params(), src=0)
        model.mark_params_modified()
        # ... but DIFFERENT timestep / noise streams: train_step draws t and the noise from torch's default CPU / CUDA
        # generators, whose seed is the same constant in every fresh process.  (The harness mixes the epoch in on
        # resume, see ModelInterface._run_epochs.)
        torch.manual_seed(1234 + rank)

    diffusion_model = DDIMDiffusionModel(
        model_class=model, num_timesteps=config["model"]["num_timesteps"],
        beta_schedule_type=config["model"]["beta_schedule_type"], pred_type=config["model"]["pred_type"],
        auto_normalize=config["model"]["auto_normalize"], ms1_loss_weight=config["model"]["ms1_loss_weight"],
        device=device)
    diffusion_model.micro_batch = int(os.environ.get("DQUARTIC_MICRO_BATCH", "0")) or None
    diffusion_model.ema_decay = config["model"].get("ema_decay")
    if val_cfg is not None:
        diffusion_model.validation = ValidationSet(data_loader, val_pairs, config["model"]["num_timesteps"],
                                                   val_cfg["bands"], val_cfg["seed"], val_cfg["every_n_epochs"])

    if use_wandb and rank == 0:
        import wandb
        w = config["wandb"]
        wandb.init(project=w["wandb_project"], name=w["wandb_name"], id=w["wandb_id"], resume=w["wandb_resume"],
                   config={"architecture": w["wandb_architecture"], "dataset": w["wandb_dataset"], **config["model"]},
                   settings=wandb.Settings(start_method="fork"), mode=w["wandb_mode"])

    diffusion_model.train(data_loader, batch_size, config["model"]["num_epochs"], config["model"]["warmup_epochs"],
                          config["model"]["learning_rate"], use_wandb, checkpoint_path)

    if use_wandb and rank == 0:
        import wandb
        wandb.finish()
    if world > 1:
        torch.distributed.destroy_process_group()


def _validation_section(config, for_train):
    """The config's "validation" section range-checked with its defaults filled in, or None when it is absent."""
    if "validation" not in config:
        return None
    try:
        return check_section(config["validation"], for_train)
    except ValueError as e:
        raise click.BadParameter(str(e), param_hint="--validation-fraction / the config's validation section")


def _validation_pairs(dataset, val_cfg):
    """Hold out the config's fraction of `dataset` and draw the fixed validation pairs (host only)."""
    try:
        lo, hi = hold_out(dataset, val_cfg["fraction"])
        return validation_pairs(dataset, lo, hi, val_cfg["windows"], val_cfg["seed"])
    except ValueError as e:
        raise click.UsageError(str(e))


PREDICT_SLICE_CHUNKS = 16   # windows handed to sample_windows at a time, in chunks: bounds the pinned host buffer


def predict_to_file(diffusion_model, ms2, ms1, output, rank=0, world=1, sampler="dpm++2m", num_steps=20, seed=0,
                    chunk=32):
    """Deconvolve every window of `ms2` (N, rt, mz) conditioned on `ms1` (N, rt) into the .npy file `output`, float32
    (N, rt, mz) in the input's intensity units.  Each window is min-max scaled on its own (MS2 and MS1 separately; a
    zero range counts as 1), sampled with x_T from (seed, window index), and the prediction is scaled back with
    pred * (max - min) + min.  This process samples the block `shard_windows(N, rank, world)`: rank 0 creates the
    file, and under torch.distributed every rank writes its own slice after a barrier (no gather)."""
    n = ms2.shape[0]
    rt, mz = ms2.shape[1], ms2.shape[2]
    dev = torch.device(diffusion_model.device)
    dist = torch.distributed
    on = dist.is_available() and dist.is_initialized()
    if rank == 0:
        np.lib.format.open_memmap(output, mode="w+", dtype=np.float32, shape=(n, rt, mz)).flush()
    if on:
        dist.barrier()
    lo, hi = diffusion_model.shard_windows(n, rank, world)
    if hi > lo:
        dst = np.load(output, mmap_mode="r+")
        ms2_min = np.empty(n, dtype=np.float32)
        ms2_rng = np.empty(n, dtype=np.float32)

        def scaled(raw):
            # min and max on the host (no device sync: the previous chunk is still running), (x - min) / range in
            # float64 on the device
            flat = raw.reshape(raw.shape[0], -1)
            mn = flat.min(1).astype(np.float64)
            rng = flat.max(1).astype(np.float64) - mn
            rng[rng == 0] = 1.0
            shape = (-1,) + (1,) * (raw.ndim - 1)
            x = torch.from_numpy(raw).to(dev).double()
            x = (x - torch.from_numpy(mn).to(dev).view(shape)) / torch.from_numpy(rng).to(dev).view(shape)
            return x.float(), mn, rng

        def cond_fn(ids):   # ids: a contiguous run of window indices (sample_windows chunks the range it is given)
            c2, mn, rng = scaled(np.ascontiguousarray(ms2[ids[0]:ids[-1] + 1]))
            ms2_min[ids[0]:ids[-1] + 1] = mn
            ms2_rng[ids[0]:ids[-1] + 1] = rng
            return c2, scaled(np.ascontiguousarray(ms1[ids[0]:ids[-1] + 1]))[0]

        step = PREDICT_SLICE_CHUNKS * chunk
        buf = torch.empty((min(step, hi - lo), rt, mz), dtype=torch.float32).pin_memory()
        for s in range(lo, hi, step):
            e = min(s + step, hi)
            _, maps = diffusion_model.sample_windows(list(range(s, e)), cond_fn, seed=seed, num_steps=num_steps,
                                                     chunk=chunk, rank=0, world=1, out=buf[:e - s], sampler=sampler)
            m = maps.numpy()
            m *= ms2_rng[s:e, None, None]
            m += ms2_min[s:e, None, None]
            dst[s:e] = m
        dst.flush()
        del dst
    if on:
        dist.barrier()


@cli.command()
@click.argument("config-path", type=click.Path(exists=True, dir_okay=False), required=True)
@click.option("--checkpoint-path", required=True, type=click.Path(exists=True, dir_okay=False),
              help="Checkpoint written by `dquartic train`")
@click.option("--ms2-data-path", required=True, type=click.Path(exists=True, dir_okay=False),
              help="MS2 mixtures, .npy of shape (N, rt, mz), any numeric dtype")
@click.option("--ms1-data-path", required=True, type=click.Path(exists=True, dir_okay=False),
              help="MS1 conditioning, .npy of shape (N, rt)")
@click.option("--output", required=True, type=click.Path(dir_okay=False),
              help="Output .npy: the deconvolved maps, float32 (N, rt, mz), in input order and intensity units")
@click.option("--sampler", default="dpm++2m", show_default=True, type=click.Choice(SAMPLERS))
@click.option("--num-steps", default=20, show_default=True, type=int, help="Denoiser evaluations per window")
@click.option("--seed", default=0, show_default=True, type=int, help="x_T of a window depends on (seed, its index)")
@click.option("--chunk", default=32, show_default=True, type=click.IntRange(min=1), help="Windows per sampler batch")
@click.option("--weights", default="auto", show_default=True, type=click.Choice(["auto", "ema", "model"]),
              help="auto: the weight EMA when the checkpoint has one, else the trained weights")
def predict(config_path, checkpoint_path, ms2_data_path, ms1_data_path, output, sampler, num_steps, seed, chunk,
            weights):
    """
    Deconvolve the MS2 windows of a DIA run with a trained checkpoint.
    """
    config = load_train_config(config_path)
    m = config["model"]
    T = int(m["num_timesteps"])
    ms2 = np.load(ms2_data_path, mmap_mode="r")
    ms1 = np.load(ms1_data_path, mmap_mode="r")
    if ms2.ndim != 3 or ms1.ndim != 2:
        raise click.UsageError(f"expected MS2 (N, rt, mz) and MS1 (N, rt), got {ms2.shape} and {ms1.shape}")
    if ms2.shape[0] != ms1.shape[0]:
        raise click.UsageError(f"{ms2.shape[0]} MS2 windows but {ms1.shape[0]} MS1 chromatograms")
    if ms2.shape[2] != m["UNet1d"]["downsample_dim"]:
        raise click.UsageError(f"MS2 m/z axis is {ms2.shape[2]}, the model's downsample_dim is "
                               f"{m['UNet1d']['downsample_dim']}")
    if ms2.shape[1] != ms1.shape[1]:
        raise click.UsageError(f"MS2 has {ms2.shape[1]} retention-time points, MS1 has {ms1.shape[1]}")
    if not 2 <= num_steps <= T:
        raise click.BadParameter(f"needs 2 <= num-steps <= {T}, got {num_steps}", param_hint="--num-steps")
    ck = torch.load(checkpoint_path, map_location="cpu", mmap=True, weights_only=False)
    if weights == "ema" and "ema_state_dict" not in ck:
        raise click.UsageError(f"{checkpoint_path} has no ema_state_dict (train with --ema-decay to keep one)")
    use_ema = weights == "ema" or (weights == "auto" and "ema_state_dict" in ck)

    rank, world, local = _init_distributed()
    if rank == 0:
        click.echo(f"Info: sampling {ms2.shape[0]} windows with {sampler} x {num_steps} steps, "
                   f"{'EMA' if use_ema else 'trained'} weights of {checkpoint_path}")
    if not torch.cuda.is_available():
        raise RuntimeError("the B200 build of dquartic has no CPU sampling path")
    device = torch.device("cuda", local)
    net = _unet_from_config(config)
    net.load_state_dict(ck["ema_state_dict"] if use_ema else ck["model_state_dict"])
    del ck
    diffusion_model = DDIMDiffusionModel(
        model_class=net.to(device), num_timesteps=T, beta_schedule_type=m["beta_schedule_type"],
        pred_type=m["pred_type"], auto_normalize=m["auto_normalize"], device=device)
    predict_to_file(diffusion_model, ms2, ms1, output, rank, world, sampler, num_steps, seed, chunk)
    if world > 1:
        torch.distributed.destroy_process_group()
    if rank == 0:
        click.echo(f"Info: wrote {output}")


def evaluate_model(diffusion_model, vset, sampler="dpm++2m", num_steps=20, seed=0, chunk=32, rank=None, world=None):
    """Score the current weights of `diffusion_model` on the validation set `vset`: the held-out denoising loss per band
    (`validate`) and, unless `num_steps` is 0, the maps `sampler` draws in `num_steps` steps against the clean maps
    (`score_samples`).  Every rank of a process group must call it; each returns the full result.  Returns a
    JSON-ready dict {"loss_by_band", "val_loss"[, "samplers": {"<sampler>@<steps>": {"mean", "per_window"}}]}."""
    v = diffusion_model.validate(vset, chunk=chunk, rank=rank, world=world)
    out = {"loss_by_band": [float(x) for x in v["loss_by_band"]], "val_loss": v["val_loss"]}
    if num_steps:
        s = diffusion_model.score_samples(vset, sampler=sampler, num_steps=num_steps, seed=seed, chunk=chunk,
                                          rank=rank, world=world)
        out["samplers"] = {f"{sampler}@{num_steps}": {
            "mean": s["mean"], "per_window": {k: [float(x) for x in a] for k, a in s["per_window"].items()}}}
    return out


@cli.command()
@click.argument("config-path", type=click.Path(exists=True, dir_okay=False), required=True)
@click.option("--checkpoint-path", required=True, type=click.Path(exists=True, dir_okay=False),
              help="Checkpoint written by `dquartic train`")
@click.option("--parquet_directory", default=None, help="Directory of Parquet slices, overrides config file")
@click.option("--ms2-data-path", default=None, help="Path to MS2 data, overrides config file")
@click.option("--ms1-data-path", default=None, help="Path to MS1 data, overrides config file")
@click.option("--validation-fraction", default=None, type=float,
              help="Held-out fraction of the slices (0 < f <= 1; 1 scores whole files), overrides validation.fraction "
                   "of the config file")
@click.option("--weights", default="auto", show_default=True, type=click.Choice(["auto", "ema", "model", "both"]),
              help="auto: the weight EMA when the checkpoint has one, else the trained weights; both: each in turn")
@click.option("--sampler", default="dpm++2m", show_default=True, type=click.Choice(SAMPLERS))
@click.option("--num-steps", default=20, show_default=True, type=int,
              help="Denoiser evaluations per sampled map; 0: the denoising loss only")
@click.option("--seed", default=0, show_default=True, type=int, help="x_T of a window depends on (seed, its index)")
@click.option("--chunk", default=32, show_default=True, type=click.IntRange(min=1), help="Windows per batch")
@click.option("--output", default=None, type=click.Path(dir_okay=False), help="JSON file (default: stdout)")
def evaluate(config_path, checkpoint_path, parquet_directory, ms2_data_path, ms1_data_path, validation_fraction, weights,
             sampler, num_steps, seed, chunk, output):
    """
    Score a checkpoint on the held-out validation mixtures: denoising loss per timestep band and sampled-map scores.
    """
    import json

    config = load_train_config(config_path, parquet_directory=parquet_directory, ms2_data_path=ms2_data_path,
                               ms1_data_path=ms1_data_path, validation_fraction=validation_fraction)
    val_cfg = _validation_section(config, for_train=False)
    if val_cfg is None:
        raise click.UsageError("the config has no validation section: pass --validation-fraction")
    m = config["model"]
    T = int(m["num_timesteps"])
    if num_steps != 0 and not 2 <= num_steps <= T:
        raise click.BadParameter(f"needs 0 or 2 <= num-steps <= {T}, got {num_steps}", param_hint="--num-steps")
    ck = torch.load(checkpoint_path, map_location="cpu", mmap=True, weights_only=False)
    has_ema = "ema_state_dict" in ck
    if weights in ("ema", "both") and not has_ema:
        raise click.UsageError(f"{checkpoint_path} has no ema_state_dict (train with --ema-decay to keep one)")
    names = {"auto": ["ema" if has_ema else "model"], "ema": ["ema"], "model": ["model"], "both": ["model", "ema"]}[weights]
    dataset = DIAMSDataset(config["data"]["parquet_directory"], config["data"]["ms2_data_path"],
                           config["data"]["ms1_data_path"], normalize=config["data"]["normalize"])
    if dataset.ms2_data.shape[2] != m["UNet1d"]["downsample_dim"]:
        raise click.UsageError(f"MS2 m/z axis is {dataset.ms2_data.shape[2]}, the model's downsample_dim is "
                               f"{m['UNet1d']['downsample_dim']}")
    pairs = _validation_pairs(dataset, val_cfg)

    rank, world, local = _init_distributed()
    if not torch.cuda.is_available():
        raise RuntimeError("the B200 build of dquartic has no CPU evaluation path")
    device = torch.device("cuda", local)
    loader = DeviceBatchLoader(dataset, 1, device, pool="hbm")
    vset = ValidationSet(loader, pairs, T, val_cfg["bands"], val_cfg["seed"], val_cfg["every_n_epochs"])
    net = _unet_from_config(config).to(device)
    diffusion_model = DDIMDiffusionModel(
        model_class=net, num_timesteps=T, beta_schedule_type=m["beta_schedule_type"], pred_type=m["pred_type"],
        auto_normalize=m["auto_normalize"], device=device)
    result = {"checkpoint": checkpoint_path, "weights": names, "windows": vset.windows, "bands": vset.bands,
              "results": {}}
    for name in names:
        net.load_state_dict(ck["ema_state_dict"] if name == "ema" else ck["model_state_dict"])
        result["results"][name] = evaluate_model(diffusion_model, vset, sampler, num_steps, seed, chunk)
        if rank == 0:
            click.echo(f"Info: {name} weights: val_loss={result['results'][name]['val_loss']}", err=True)
    if rank == 0:
        text = json.dumps(result)
        if output is None:
            click.echo(text)
        else:
            with open(output, "w") as f:
                f.write(text + "\n")
    if world > 1:
        torch.distributed.destroy_process_group()


@cli.command()
@click.argument("config-path", type=click.Path(exists=False), default="dquartic_train_config.json", required=False)
def generate_config(config_path):
    """
    Generate a default training config file.
    """
    generate_train_config(config_path)
    click.echo(f"Info: wrote {config_path}")


if __name__ == "__main__":
    cli()
