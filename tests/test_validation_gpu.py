"""Held-out validation on the GPU: dq_map_scores against the float64 oracle and its bit-identity, `denoising_loss` on an
analytic Gaussian problem, `validate` rank by rank and under the weight EMA, and training + `dquartic evaluate` end to
end on the tiny denoiser."""
import json
import math
import re

import numpy as np
import pytest
import torch

import _eval_oracle as EO
from _util import TINY, make_net

pytestmark = pytest.mark.gpu


def _scores(p, g):
    from dquartic.model.model_interface import ModelInterface
    return ModelInterface.map_scores(p, g)


def _placed(a, off):
    """`a` (numpy) copied to the device at element offset `off` of a fresh buffer (off 1: unaligned base pointer)."""
    t = torch.from_numpy(np.ascontiguousarray(a)).reshape(-1)
    buf = torch.empty(t.numel() + 4, device="cuda")
    view = buf[off:off + t.numel()]
    view.copy_(t)
    return view.view(a.shape)


# ------------------------------------------------------------------------------------------ kernel
@pytest.mark.parametrize("rt", [34, 136])
@pytest.mark.parametrize("mz,off", [(2048, 0), (2048, 1), (1030, 0), (321, 1), (5, 0)])
def test_map_scores_match_the_float64_oracle(rt, mz, off):
    """fp32 inputs are exact in float64, so the only differences are float64 summation order (and the kernel's shifted
    one-pass column statistics): every slot agrees to 1e-9 of its magnitude."""
    p, g = EO.sparse_maps(3, rt, mz, seed=rt + mz + off)
    got = _scores(_placed(p, off), _placed(g, off)).cpu().numpy()
    want = EO.map_sums(p, g)
    mag = np.abs(want)
    mag[:, 7] = want[:, 8]                # |sum w r| <= sum w
    np.testing.assert_array_less(np.abs(got - want), 1e-9 * mag + 1e-12)
    assert (want[:, 8] > 0).all() and (want[:, 8] < g.astype(np.float64).sum((1, 2))).all()   # column 1 skipped


def test_map_scores_are_bit_identical_alone_in_a_batch_and_on_rerun():
    p, g = EO.sparse_maps(6, 34, 4000, seed=9)
    P, G = torch.from_numpy(p).cuda(), torch.from_numpy(g).cuda()
    batch = _scores(P, G)
    assert torch.equal(batch, _scores(P, G))
    for w in range(6):
        assert torch.equal(_scores(P[w:w + 1].clone(), G[w:w + 1].clone())[0], batch[w]), w
    assert torch.equal(_scores(P[2:5], G[2:5]), batch[2:5])
    # unaligned copies take the scalar loads: same sums, bit for bit
    assert torch.equal(_scores(_placed(p, 1), _placed(g, 1)), batch)


# ------------------------------------------------------------------------------------------ denoising loss
def _ab():
    import dquartic_oracle as O
    return O.schedule_tables(1000, "cosine")[2].numpy().astype(np.float64)


class _GaussNet(torch.nn.Module):
    """Optimal denoiser of elementwise Gaussian data x0 ~ N(mu, s^2) (tests/_ode_oracle.py) as the network."""

    def __init__(self, mu, s2, ab, pred_type):
        super().__init__()
        self.mu, self.s2, self.ab, self.pred_type = mu, s2, torch.from_numpy(ab).cuda(), pred_type

    def forward(self, x, t, init_cond=None, attn_cond=None):
        a2 = self.ab[t].view(-1, 1, 1)
        a = a2.sqrt()
        D = self.mu + a * self.s2 * (x.double() - a * self.mu) / (a2 * self.s2 + 1 - a2)
        return (D if self.pred_type == "x0" else (x.double() - a * D) / (1 - a2).sqrt()).float()


@pytest.mark.parametrize("pred_type", ["eps", "x0"])
def test_denoising_loss_of_the_optimal_gaussian_denoiser(pred_type):
    """E|eps - eps_hat|^2 = mean(a^2 s^2 / (a^2 s^2 + sigma^2)) and E|x0 - x0_hat|^2 = mean(s^2 sigma^2 / (...)) per
    element; the per-element squared errors are Gaussian squares, so the mean of 1e5 of them is within 5 standard
    deviations sqrt(2 sum v^2) / n of the expectation."""
    from dquartic.model.model import DDIMDiffusionModel
    from dquartic.utils.validation import band_timesteps

    ab = _ab()
    shape = (25, 4000)
    rng = np.random.default_rng(3)
    mu = torch.from_numpy(rng.uniform(-1, 1, shape)).cuda()
    s2 = torch.from_numpy(rng.uniform(0.05, 0.5, shape) ** 2).cuda()
    d = DDIMDiffusionModel(torch.nn.Identity(), device="cuda", pred_type=pred_type, auto_normalize=False)
    d.model = _GaussNet(mu, s2, ab, pred_type)
    bands = band_timesteps(1000, 10)
    g = torch.Generator(device="cuda").manual_seed(1)
    x0 = (mu + s2.sqrt() * torch.randn((10,) + shape, device="cuda", generator=g, dtype=torch.float64)).float()
    noise = torch.randn((10,) + shape, device="cuda", generator=g)
    got = d.denoising_loss(x0, None, None, torch.tensor(bands, device="cuda"), noise).cpu().numpy()
    assert got.dtype == np.float64 and got.shape == (10,)
    s2n = s2.cpu().numpy()
    n = s2n.size
    for k, t in enumerate(bands):
        a2 = ab[t]
        v = a2 * s2n / (a2 * s2n + 1 - a2) if pred_type == "eps" else s2n * (1 - a2) / (a2 * s2n + 1 - a2)
        bound = 5 * math.sqrt(2 * float((v * v).sum())) / n
        assert abs(got[k] - v.mean()) < bound, (t, got[k], v.mean(), bound)


# ------------------------------------------------------------------------------------------ validate
def _pool_loader(tmp_path, n=16, seed=0):
    from dquartic.utils.data_loader import DeviceBatchLoader, DIAMSDataset
    from dquartic.utils.synthetic import synth_pool

    ms2, ms1 = synth_pool(n, 6, 320, seed=seed, density=0.2)
    np.save(tmp_path / "ms2.npy", ms2)
    np.save(tmp_path / "ms1.npy", ms1)
    ds = DIAMSDataset(ms2_file=str(tmp_path / "ms2.npy"), ms1_file=str(tmp_path / "ms1.npy"), normalize="minmax")
    return ds, DeviceBatchLoader(ds, 4, "cuda", pool="hbm")


def _vset(tmp_path, windows=5, bands=3, fraction=0.5):
    from dquartic.utils.validation import ValidationSet, hold_out, validation_pairs

    ds, loader = _pool_loader(tmp_path)
    lo, hi = hold_out(ds, fraction)
    return ValidationSet(loader, validation_pairs(ds, lo, hi, windows, seed=2), 1000, bands=bands, seed=4)


@pytest.mark.parametrize("pred_type", ["eps", "x0"])
def test_validate_rank_by_rank_is_bit_identical_to_one_rank(tmp_path, pred_type):
    from dquartic.model.model import DDIMDiffusionModel

    vset = _vset(tmp_path)
    d = DDIMDiffusionModel(make_net(seed=5)[0], device="cuda", pred_type=pred_type)
    one = d.validate(vset, chunk=4, rank=0, world=1)
    assert one["per_window"].shape == (5, 3) and one["windows"] == (0, 5) and one["bands"] == [166, 500, 833]
    assert np.isfinite(one["per_window"]).all() and (one["per_window"] > 0).all()
    lw = d.loss_weight.double().cpu().numpy()[one["bands"]]
    assert one["val_loss"] == float(np.mean(lw * one["per_window"].mean(0)))
    for world, chunk in ((2, 4), (4, 3), (1, 64)):
        parts = [d.validate(vset, chunk=chunk, rank=r, world=world) for r in range(world)]
        assert [p["windows"] for p in parts] == [d.shard_windows(5, r, world) for r in range(world)]
        cat = np.concatenate([p["per_window"] for p in parts])
        assert np.array_equal(cat, one["per_window"]), (world, chunk)
    # fixed noise: a second pass is the same, and the noise of window w is the sample_windows x_T of window w
    assert np.array_equal(d.validate(vset, chunk=4)["per_window"], one["per_window"])
    xT = torch.empty_like(vset.noise[3]).normal_(generator=torch.Generator(device="cuda").manual_seed(d.window_seed(4, 3)))
    assert torch.equal(xT, vset.noise[3])


def test_validate_inside_ema_weights_equals_a_fresh_network_with_the_ema(tmp_path):
    from dquartic.model.model import DDIMDiffusionModel

    vset = _vset(tmp_path, windows=4, bands=2)
    net, _ = make_net(seed=6)
    d = DDIMDiffusionModel(net, device="cuda")
    d.ema_decay = 0.5
    d._prepare_training(1e-3)
    n = net.n_trainable_flat
    for k in range(3):
        net.flat_grads()[:n].copy_(1e-1 * torch.randn(n, device="cuda",
                                                      generator=torch.Generator(device="cuda").manual_seed(k)))
        d.optimizer.step(max_grad_norm=d.max_grad_norm)
    live = d.validate(vset, chunk=3)
    with d.ema_weights():
        ema = d.validate(vset, chunk=3)
    fresh, _ = make_net(seed=0)
    fresh.load_state_dict(d.optimizer.ema_state_dict())
    ref = DDIMDiffusionModel(fresh, device="cuda").validate(vset, chunk=8)
    assert np.array_equal(ema["per_window"], ref["per_window"]) and ema["val_loss"] == ref["val_loss"]
    assert ema["val_loss"] != live["val_loss"]
    assert np.array_equal(d.validate(vset, chunk=3)["per_window"], live["per_window"])   # live weights are back


# ------------------------------------------------------------------------------------------ train + evaluate
def _run(args):
    from click.testing import CliRunner
    from dquartic import cli

    res = CliRunner().invoke(cli.cli, args)
    assert res.exit_code == 0, (res.output, res.exception)
    return res.output


@pytest.fixture(scope="module")
def trained(tmp_path_factory):
    """`dquartic train` for 2 epochs on 16 slices of 6 x 320 with 4 held out (6 validation windows, 4 bands) and the
    weight EMA on, and once more without validation."""
    from dquartic.utils.config_loader import default_train_config
    from dquartic.utils.synthetic import synth_pool

    tmp = tmp_path_factory.mktemp("val_train")
    ms2, ms1 = synth_pool(16, 6, 320, seed=11, density=0.2)
    np.save(tmp / "ms2.npy", ms2)
    np.save(tmp / "ms1.npy", ms1)
    cfg = default_train_config()
    cfg["model"]["UNet1d"].update({k: TINY[k] for k in cfg["model"]["UNet1d"]})
    cfg["model"].update(batch_size=4, num_epochs=2, warmup_epochs=1, checkpoint_path=str(tmp / "val" / "best.ckpt"))
    cfg["wandb"]["use_wandb"] = False
    cfg["data"].update(parquet_directory=None, ms2_data_path=str(tmp / "ms2.npy"), ms1_data_path=str(tmp / "ms1.npy"))
    cfg["validation"] = {"fraction": 0.5, "windows": 6, "bands": 4, "seed": 1}
    (tmp / "cfg.json").write_text(json.dumps(cfg))
    (tmp / "val").mkdir()
    (tmp / "plain").mkdir()
    out = _run(["train", "--ema-decay", "0.9", "--validation-fraction", "0.25", str(tmp / "cfg.json")])
    plain_cfg = dict(cfg)
    plain_cfg.pop("validation")
    plain_cfg["model"] = dict(cfg["model"], checkpoint_path=str(tmp / "plain" / "best.ckpt"))
    (tmp / "plain.json").write_text(json.dumps(plain_cfg))
    _run(["train", str(tmp / "plain.json")])
    return tmp, out


def test_training_selects_the_best_checkpoint_by_the_ema_validation_loss(trained):
    tmp, out = trained
    lines = re.findall(r"\[Validation\] Epoch=(\d+), val_loss=(\S+), ema_val_loss=(\S+)", out)
    assert [int(e) for e, _, _ in lines] == [1, 2], out
    live = [float(v) for _, v, _ in lines]
    ema = [float(v) for _, _, v in lines]
    assert all(math.isfinite(v) for v in live + ema)
    best = torch.load(str(tmp / "val" / "best.ckpt"), weights_only=False)
    latest = torch.load(str(tmp / "val" / "dquartic_latest_checkpoint.ckpt"), weights_only=False)
    assert best["best_loss"] == min(ema) and best["val_loss"] == best["best_loss"]
    assert best["epoch"] == int(np.argmin(ema))
    assert latest["val_loss"] == ema[-1] and latest["best_loss"] == min(ema) and latest["epoch"] == 1
    plain = torch.load(str(tmp / "plain" / "dquartic_latest_checkpoint.ckpt"), weights_only=False)
    assert "val_loss" not in plain and "val_loss" not in torch.load(str(tmp / "plain" / "best.ckpt"), weights_only=False)


def test_evaluate_reproduces_the_last_validation_exactly(trained):
    tmp, out = trained
    lines = re.findall(r"\[Validation\] Epoch=2, val_loss=(\S+), ema_val_loss=(\S+)", out)
    live, ema = float(lines[0][0]), float(lines[0][1])
    res = tmp / "eval.json"
    _run(["evaluate", "--checkpoint-path", str(tmp / "val" / "dquartic_latest_checkpoint.ckpt"), "--num-steps", "0",
          "--weights", "both", "--validation-fraction", "0.25", "--output", str(res), str(tmp / "cfg.json")])
    r = json.loads(res.read_text())
    assert r["weights"] == ["model", "ema"] and r["windows"] == 6 and r["bands"] == [125, 375, 625, 875]
    assert r["results"]["model"]["val_loss"] == live
    assert r["results"]["ema"]["val_loss"] == ema
    assert "samplers" not in r["results"]["model"]


def test_evaluate_with_a_sampler_scores_every_window(trained):
    tmp, _ = trained
    res = tmp / "eval_dpm.json"
    _run(["evaluate", "--checkpoint-path", str(tmp / "val" / "best.ckpt"), "--num-steps", "4", "--chunk", "4",
          "--validation-fraction", "0.25", "--output", str(res), str(tmp / "cfg.json")])
    r = json.loads(res.read_text())
    assert r["weights"] == ["ema"]
    s = r["results"]["ema"]["samplers"]["dpm++2m@4"]
    for k in ("cosine", "rmse", "spectral_angle", "xic_corr"):
        assert len(s["per_window"][k]) == 6 and all(math.isfinite(v) for v in s["per_window"][k]), k
        assert s["mean"][k] == pytest.approx(float(np.mean(s["per_window"][k])), rel=1e-12)
    assert all(-1 <= v <= 1 for v in s["per_window"]["cosine"] + s["per_window"]["xic_corr"])
