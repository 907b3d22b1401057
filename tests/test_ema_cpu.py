"""CPU (no GPU needed): the host side of the weight EMA — config key and CLI option, argument checks, decay warm-up."""
import json

import pytest
import torch

from _util import TINY

from dquartic.model.model_interface import FusedAdamW, ModelInterface
from dquartic.model.unet1d import UNet1d
from dquartic.utils.config_loader import generate_train_config, load_train_config


def _net():
    return UNet1d(dim=TINY["dim"], channels=1, dim_mults=tuple(TINY["dim_mults"]), conditional=True,
                  init_cond_channels=1, attn_cond_channels=1, downsample_dim=TINY["downsample_dim"], simple=True)


def test_config_ema_decay_is_optional_and_overridable(tmp_path):
    p = str(tmp_path / "cfg.json")
    generate_train_config(p)
    cfg = load_train_config(p)
    assert "ema_decay" not in cfg["model"] and cfg["model"].get("ema_decay") is None     # absent: off
    assert load_train_config(p, ema_decay=None)["model"].get("ema_decay") is None
    assert load_train_config(p, ema_decay=0.999)["model"]["ema_decay"] == 0.999
    raw = json.load(open(p))
    raw["model"]["ema_decay"] = 0.99
    p2 = str(tmp_path / "cfg_ema.json")
    json.dump(raw, open(p2, "w"))
    assert load_train_config(p2)["model"]["ema_decay"] == 0.99
    assert load_train_config(p2, ema_decay=None)["model"]["ema_decay"] == 0.99     # None does not override
    assert load_train_config(p2, ema_decay=0.9999)["model"]["ema_decay"] == 0.9999  # the CLI value wins


def test_cli_train_has_ema_decay_option():
    from click.testing import CliRunner
    from dquartic.cli import cli

    r = CliRunner().invoke(cli, ["train", "--help"])
    assert r.exit_code == 0 and "--ema-decay" in r.output


@pytest.mark.parametrize("bad", [0, 0.0, 1, 1.0, -0.5, 1.5, float("nan")])
def test_fused_adamw_rejects_ema_decay_outside_open_unit_interval(bad):
    with pytest.raises(ValueError):
        FusedAdamW(_net(), ema_decay=bad)


def test_fused_adamw_ema_off_by_default_and_accepts_valid_decay():
    net = _net()
    assert FusedAdamW(net).ema_decay is None
    opt = FusedAdamW(net, ema_decay=0.999)
    assert opt.ema_decay == 0.999 and opt.ema_updates == 0
    assert set(opt.state_dict()) == {"state", "param_groups"}


def test_ema_decay_warmup_sequence():
    for decay in (0.5, 0.9, 0.999, 0.9999):
        for k in range(0, 20000, 7):
            assert FusedAdamW.ema_beta(decay, k) == min(decay, (1 + k) / (10 + k))
    assert FusedAdamW.ema_beta(0.999, 0) == 0.1
    assert FusedAdamW.ema_beta(0.999, 9000) == 0.999 and FusedAdamW.ema_beta(0.999, 8980) < 0.999


def test_ema_decay_needs_the_flat_buffer_api():
    mi = ModelInterface(device=torch.device("cpu"))
    mi.model = torch.nn.Linear(3, 2)
    mi.ema_decay = 0.999
    with pytest.raises(ValueError):
        mi._set_optimizer(1e-3)
    mi.ema_decay = None
    mi._set_optimizer(1e-3)
    assert isinstance(mi.optimizer, torch.optim.AdamW)
    with pytest.raises(RuntimeError):
        with mi.ema_weights():
            pass
