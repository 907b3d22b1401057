"""`dquartic` command line — same commands and options as the reference (/root/reference/dquartic/cli.py:26-188):
`dquartic train CONFIG [--parquet_directory --ms2-data-path --ms1-data-path --batch-size --checkpoint-path
--use-wandb --threads]`, `dquartic generate-config`.  `--ema-decay` (model.ema_decay in the config) keeps an exponential
moving average of the weights in the checkpoints.  Differences: `--batch-size/--threads` are cast to int (the
reference passes strings to DataLoader and fails, SURVEY.md §5); under torchrun (RANK/WORLD_SIZE in the
environment) each rank binds one GPU, joins an NCCL process group and trains a batch shard;
`generate-train-data` (offline ETL) is out of scope.
"""
import ast
import os

import click
import torch

from .model.model import DDIMDiffusionModel
from .model.unet1d import UNet1d
from .utils.config_loader import generate_train_config, load_train_config
from .utils.data_loader import DeviceBatchLoader, DIAMSDataset


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
def train(config_path, parquet_directory, ms2_data_path, ms1_data_path, batch_size, checkpoint_path, use_wandb, threads,
          ema_decay):
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
                               use_wandb=use_wandb, threads=threads, ema_decay=ema_decay)
    batch_size = int(config["model"]["batch_size"])
    checkpoint_path = config["model"]["checkpoint_path"]
    use_wandb = config["wandb"]["use_wandb"]

    if not torch.cuda.is_available():
        raise RuntimeError("the B200 build of dquartic has no CPU training path")
    device = torch.device("cuda", local)
    dataset = DIAMSDataset(config["data"]["parquet_directory"], config["data"]["ms2_data_path"],
                           config["data"]["ms1_data_path"], normalize=config["data"]["normalize"])
    if world > 1:
        import random
        random.seed(1234 + rank)  # each rank draws its own pairs, like DataLoader workers do in the reference
    per_rank = max(1, batch_size // world)
    data_loader = DeviceBatchLoader(dataset, per_rank, device, pool="hbm",
                                    batches_per_epoch=(len(dataset) + batch_size - 1) // batch_size)

    if config["model"]["use_model"] == "UNet1d":
        u = config["model"]["UNet1d"]
        model = UNet1d(dim=u["dim"], channels=u["channels"], dim_mults=tuple(u["dim_mults"]),
                       conditional=u["conditional"], init_cond_channels=u["init_cond_channels"],
                       attn_cond_channels=u["attn_cond_channels"], tfer_dim_mult=u["tfer_dim_mult"],
                       downsample_dim=u["downsample_dim"], simple=u["simple"]).to(device)
    elif config["model"]["use_model"] == "CustomTransformer":
        raise NotImplementedError("CustomTransformer is dead code under the reference's DDIM API (SURVEY.md finding 2)")
    else:
        raise ValueError(f"Invalid model class: {config['model']['use_model']}")
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
