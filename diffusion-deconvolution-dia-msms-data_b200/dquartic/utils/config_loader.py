"""Training-config loader — same JSON schema and override rules as the reference
(/root/reference/dquartic/utils/config_loader.py:4-57, dquartic_train_config.json): a CLI option overrides its
config entry only when it is not None.  `generate_train_config` writes the reference's default schema."""
import json

_DATA_KEYS = ("parquet_directory", "ms2_data_path", "ms1_data_path")
_OVERRIDES = {
    "parquet_directory": ("data", "parquet_directory"),
    "ms2_data_path": ("data", "ms2_data_path"),
    "ms1_data_path": ("data", "ms1_data_path"),
    "batch_size": ("model", "batch_size"),
    "checkpoint_path": ("model", "checkpoint_path"),
    "use_wandb": ("wandb", "use_wandb"),
    "ema_decay": ("model", "ema_decay"),   # optional key (absent: no weight EMA), not part of the default schema
}


def load_train_config(config_path: str, **kwargs):
    with open(config_path, "r") as f:
        cfg = json.load(f)
    for k in _DATA_KEYS:
        cfg["data"].setdefault(k, None)
    for key, (sect, name) in _OVERRIDES.items():
        if kwargs.get(key) is not None:
            cfg[sect][name] = kwargs[key]
    if kwargs.get("threads") is not None:
        cfg["threads"] = kwargs["threads"]
    if kwargs.get("validation_fraction") is not None:   # optional section, absent from the default schema
        cfg.setdefault("validation", {})["fraction"] = kwargs["validation_fraction"]
    return cfg


def default_train_config():
    return {
        "data": {"parquet_directory": "data/", "ms2_data_path": None, "ms1_data_path": None, "normalize": "minmax"},
        "model": {
            "checkpoint_path": "best_model.ckpt", "num_epochs": 10000, "warmup_epochs": 5, "batch_size": 1,
            "learning_rate": 0.00001, "num_timesteps": 1000, "beta_schedule_type": "cosine", "pred_type": "eps",
            "auto_normalize": True, "ms1_loss_weight": 0.0, "use_model": "UNet1d",
            "CustomTransformer": {"input_dim": 40000, "hidden_dim": 1024, "num_heads": 8, "num_layers": 8},
            "UNet1d": {"dim": 4, "channels": 1, "dim_mults": [1, 2, 2, 3, 3, 4, 4], "conditional": True,
                       "init_cond_channels": 1, "attn_cond_channels": 1, "tfer_dim_mult": 620,
                       "downsample_dim": 40000, "simple": True},
        },
        "wandb": {"use_wandb": True, "wandb_project": "dquartic", "wandb_name": None, "wandb_id": None,
                  "wandb_resume": None, "wandb_architecture": "DDIM(UNet1d)", "wandb_dataset": "MS2",
                  "wandb_mode": "offline"},
        "threads": 4,
    }


def generate_train_config(config_path: str):
    with open(config_path, "w") as f:
        json.dump(default_train_config(), f, indent=4)
