"""Held-out validation on the host: timestep bands, the hold-out split and the training pair stream, the fixed
validation pairs, the optional config section, `dquartic evaluate` / `train` options and argument checks, and the float64
oracle of the map scores with `finalize_scores`.  No GPU needed."""
import json
import math
import random

import numpy as np
import pytest
import torch

import _eval_oracle as EO
from dquartic.utils.config_loader import default_train_config, generate_train_config, load_train_config
from dquartic.utils.data_loader import DeviceBatchLoader, DIAMSDataset
from dquartic.utils.validation import (band_timesteps, check_section, count_pairs, finalize_scores, hold_out,
                                       validation_pairs)


def test_band_timesteps_are_stratum_centres():
    assert band_timesteps(1000, 10) == [50, 150, 250, 350, 450, 550, 650, 750, 850, 950]
    assert band_timesteps(1000, 1) == [500]
    assert band_timesteps(1000, 3) == [166, 500, 833]
    assert band_timesteps(7, 7) == list(range(7))


def _npy_dataset(tmp_path, n, rt=3, mz=8):
    rng = np.random.default_rng(n)
    np.save(tmp_path / "ms2.npy", rng.integers(0, 50, (n, rt, mz)).astype(np.int32))
    np.save(tmp_path / "ms1.npy", rng.integers(1, 50, (n, rt)).astype(np.int32))
    return DIAMSDataset(ms2_file=str(tmp_path / "ms2.npy"), ms1_file=str(tmp_path / "ms1.npy"), normalize="minmax")


def _reference_draw_pair(n, used):
    """The reference's rejection loop (data_loader.py:111-125) as it was, over all n slices."""
    while True:
        i1 = random.randint(0, n - 1)
        i2 = random.randint(0, n - 1)
        if i1 == i2:
            continue
        pair = tuple(sorted((i1, i2)))
        if pair in used:
            continue
        used.add(pair)
        return i1, i2


def test_no_split_keeps_the_pair_stream(tmp_path):
    ds = _npy_dataset(tmp_path, 20)
    assert ds.n_train == 20
    random.seed(3)
    got = [ds.draw_pair() for _ in range(150)]
    random.seed(3)
    used = set()
    assert got == [_reference_draw_pair(20, used) for _ in range(150)]


def test_held_out_slices_are_never_drawn_for_training(tmp_path):
    ds = _npy_dataset(tmp_path, 20)
    assert hold_out(ds, 0.25) == (15, 20) and ds.n_train == 15 and len(ds) == 20
    random.seed(0)
    for _ in range(4):
        ds.reset_epoch()
        pairs = [ds.draw_pair() for _ in range(105)]      # every pair of the 15 training slices
        assert len({tuple(sorted(p)) for p in pairs}) == 105
        assert max(max(p) for p in pairs) == 14
    assert DeviceBatchLoader(ds, 4, "cpu").batches_per_epoch == 4       # from the 15 training slices
    assert DeviceBatchLoader(_npy_dataset(tmp_path, 20), 4, "cpu").batches_per_epoch == 5
    assert DeviceBatchLoader(ds, 4, "cpu").ms2.shape[0] == 20             # the pool keeps the held-out slices


@pytest.mark.parametrize("n,fraction,held", [(100, 0.07, 7), (24, 0.25, 6), (520, 0.1, 52), (10, 0.01, 1), (5, 1.0, 5)])
def test_hold_out_takes_the_ceiling_of_the_last_slices(tmp_path, n, fraction, held):
    ds = _npy_dataset(tmp_path, n)
    assert hold_out(ds, fraction) == (n - held, n)
    assert ds.n_train == (n if held == n else n - held)


def test_hold_out_needs_two_training_slices(tmp_path):
    with pytest.raises(ValueError, match="at least 2"):
        hold_out(_npy_dataset(tmp_path, 4), 0.9)


def _meta_dataset(meta):
    ds = DIAMSDataset.__new__(DIAMSDataset)
    ds.ms2_data = np.zeros((len(meta), 1, 1), np.int32)
    ds.ms1_data = np.zeros((len(meta), 1), np.int32)
    ds.used_pairs = set()
    ds.pair_meta = meta
    return ds


def test_validation_pairs_are_fixed_distinct_held_out_and_follow_the_parquet_rule():
    meta = [(i % 5, 400.0 + 25 * (i % 3)) for i in range(30)]
    ds = _meta_dataset(meta)
    lo, hi = hold_out(ds, 0.4)
    assert (lo, hi) == (18, 30)
    random.seed(5)
    state = random.getstate()
    a = validation_pairs(ds, lo, hi, 40, seed=7)
    assert random.getstate() == state                         # the global stream is untouched
    assert a == validation_pairs(ds, lo, hi, 40, seed=7)
    assert a != validation_pairs(ds, lo, hi, 40, seed=8)
    assert len({tuple(sorted(p)) for p in a}) == 40
    assert all(lo <= i < hi for p in a for i in p)
    assert all(meta[i] != meta[j] for i, j in a)
    # 12 slices, (slice index, window) repeats every 15 rows: no two held-out rows share their metadata here
    assert count_pairs(ds, lo, hi) == 66
    same = _meta_dataset([(0, 1.0)] * 4 + [(1, 1.0)] * 4)
    assert count_pairs(same, 0, 8) == 28 - 6 - 6


def test_too_few_pairs_name_both_numbers():
    ds = _meta_dataset([(i, 1.0) for i in range(24)])
    lo, hi = hold_out(ds, 0.25)
    assert count_pairs(ds, lo, hi) == 15
    assert len(validation_pairs(ds, lo, hi, 15, seed=0)) == 15
    with pytest.raises(ValueError, match=r"give 15 distinct pairs, fewer than the 16"):
        validation_pairs(ds, lo, hi, 16, seed=0)


# ------------------------------------------------------------------------------------------ config
def test_absent_section_changes_nothing_and_overrides_add_it(tmp_path):
    p = str(tmp_path / "cfg.json")
    generate_train_config(p)
    cfg = load_train_config(p)
    assert "validation" not in cfg and "validation" not in default_train_config()
    assert cfg == load_train_config(p, validation_fraction=None)
    cfg = load_train_config(p, validation_fraction=0.2)
    assert cfg["validation"] == {"fraction": 0.2}
    assert check_section(cfg["validation"], True) == {"fraction": 0.2, "windows": 64, "bands": 10, "seed": 0,
                                                      "every_n_epochs": 1}
    raw = json.load(open(p))
    raw["validation"] = {"fraction": 0.5, "windows": 8, "seed": 3}
    (tmp_path / "v.json").write_text(json.dumps(raw))
    cfg = load_train_config(str(tmp_path / "v.json"), validation_fraction=0.1)
    assert cfg["validation"] == {"fraction": 0.1, "windows": 8, "seed": 3}


@pytest.mark.parametrize("sec,for_train", [
    ({"fraction": 0.0}, True), ({"fraction": 1.0}, True), ({"fraction": 1.5}, False), ({"fraction": -0.1}, False),
    ({}, False), ({"fraction": "0.2"}, True), ({"fraction": 0.2, "windows": 0}, True),
    ({"fraction": 0.2, "bands": 2.5}, True), ({"fraction": 0.2, "every_n_epochs": 0}, True),
    ({"fraction": 0.2, "seed": -1}, True), ({"fraction": 0.2, "windows": True}, True),
    ({"fraction": 0.2, "window": 4}, True),
])
def test_out_of_range_sections_are_rejected(sec, for_train):
    with pytest.raises(ValueError):
        check_section(sec, for_train)


def test_whole_files_can_be_held_out_for_evaluation():
    assert check_section({"fraction": 1.0}, False)["fraction"] == 1.0


# ------------------------------------------------------------------------------------------ CLI
def test_help_shows_the_new_options():
    from click.testing import CliRunner
    from dquartic.cli import cli

    r = CliRunner().invoke(cli, ["train", "--help"])
    assert r.exit_code == 0 and "--validation-fraction" in r.output
    r = CliRunner().invoke(cli, ["evaluate", "--help"])
    assert r.exit_code == 0
    for opt in ("--checkpoint-path", "--validation-fraction", "--weights", "--sampler", "--num-steps", "--seed",
                "--chunk", "--output", "--ms2-data-path", "--ms1-data-path", "--parquet_directory"):
        assert opt in r.output, opt


def _evaluate_args(tmp_path, mz=320, n=12, ck=None, section=None, **extra):
    from dquartic.utils.synthetic import synth_pool

    cfg = default_train_config()
    cfg["model"]["UNet1d"]["downsample_dim"] = 320
    cfg["data"]["parquet_directory"] = None
    if section is not None:
        cfg["validation"] = section
    (tmp_path / "cfg.json").write_text(json.dumps(cfg))
    ms2, ms1 = synth_pool(n, 6, mz, seed=1)
    np.save(tmp_path / "ms2.npy", ms2)
    np.save(tmp_path / "ms1.npy", ms1)
    torch.save(ck or {"model_state_dict": {}}, tmp_path / "ck.ckpt")
    args = ["evaluate", "--checkpoint-path", str(tmp_path / "ck.ckpt"), "--ms2-data-path", str(tmp_path / "ms2.npy"),
            "--ms1-data-path", str(tmp_path / "ms1.npy"), "--output", str(tmp_path / "out.json")]
    for k, v in extra.items():
        args += [f"--{k.replace('_', '-')}", str(v)]
    return args + [str(tmp_path / "cfg.json")]


@pytest.mark.parametrize("case,kw,msg", [
    ("no_section", dict(), "no validation section"),
    ("fraction", dict(validation_fraction=1.5), "validation.fraction"),
    ("fraction0", dict(validation_fraction=0), "validation.fraction"),
    ("windows", dict(section={"fraction": 0.25, "windows": 0}), "validation.windows"),
    ("steps", dict(validation_fraction=0.5, num_steps=1), "num-steps"),
    ("steps_hi", dict(validation_fraction=0.5, num_steps=1001), "num-steps"),
    ("mz", dict(validation_fraction=0.5, mz=321), "downsample_dim is 320"),
    ("pairs", dict(section={"fraction": 0.25, "windows": 4}), "give 3 distinct pairs, fewer than the 4"),
    ("ema", dict(validation_fraction=0.5, weights="ema"), "has no ema_state_dict"),
    ("both", dict(validation_fraction=0.5, weights="both"), "has no ema_state_dict"),
    ("sampler", dict(validation_fraction=0.5, sampler="euler"), "euler"),
])
def test_evaluate_validates_inputs_before_any_cuda_call(tmp_path, monkeypatch, case, kw, msg):
    from click.testing import CliRunner
    from dquartic import cli

    def no_cuda(*a, **k):
        raise AssertionError("CUDA touched before the inputs were validated")

    monkeypatch.setattr(torch.cuda, "is_available", no_cuda)
    monkeypatch.setattr(torch.cuda, "set_device", no_cuda)
    res = CliRunner().invoke(cli.cli, _evaluate_args(tmp_path, **kw))
    assert res.exit_code == 2, (res.output, res.exception)
    assert msg in res.output, res.output
    assert not (tmp_path / "out.json").exists()


def test_train_rejects_a_bad_fraction_before_loading_data(tmp_path):
    from click.testing import CliRunner
    from dquartic import cli

    args = _evaluate_args(tmp_path)
    cfg = args[-1]
    for f in ("1.0", "0"):
        res = CliRunner().invoke(cli.cli, ["train", "--validation-fraction", f, "--ms2-data-path",
                                           str(tmp_path / "ms2.npy"), "--ms1-data-path", str(tmp_path / "ms1.npy"), cfg])
        assert res.exit_code == 2 and "validation.fraction" in res.output, res.output


# ------------------------------------------------------------------------------------------ map-score oracle
def test_identical_maps_score_perfectly():
    p, g = EO.sparse_maps(3, 6, 50, seed=0)
    sc = EO.scores(g, g)
    np.testing.assert_allclose(sc["cosine"], 1, atol=1e-14)
    assert (sc["rmse"] == 0).all()
    np.testing.assert_allclose(sc["spectral_angle"], 1, atol=1e-7)     # acos near 1 loses half the digits
    np.testing.assert_allclose(sc["xic_corr"], 1, atol=1e-14)


def test_a_positive_multiple_keeps_the_shape_scores():
    _, g = EO.sparse_maps(2, 34, 64, seed=1)
    sc = EO.scores(3.5 * g.astype(np.float64), g)
    np.testing.assert_allclose(sc["cosine"], 1, atol=1e-14)
    np.testing.assert_allclose(sc["spectral_angle"], 1, atol=1e-7)
    np.testing.assert_allclose(sc["xic_corr"], 1, atol=1e-14)
    assert (sc["rmse"] > 0.1).all()


def test_flat_predicted_column_has_r_zero_and_constant_truth_column_is_skipped():
    g = np.zeros((1, 4, 3))
    g[0, :, 0] = [0, 1, 2, 3]          # varies: weight 6
    g[0, :, 1] = 2.0                   # constant truth: skipped whatever the prediction
    g[0, :, 2] = [1, 0, 0, 1]          # varies: weight 2
    p = g.copy()
    p[0, :, 1] = [5, 0, 1, 0]
    p[0, :, 2] = 0.7                   # flat prediction: r = 0
    s = EO.map_sums(p, g)
    assert s[0, 8] == 8.0 and abs(s[0, 7] - 6.0) < 1e-14
    assert abs(EO.scores(p, g)["xic_corr"][0] - 0.75) < 1e-15
    assert EO.scores(np.ones((1, 4, 3)), np.full((1, 4, 3), 2.0))["xic_corr"][0] == 0.0   # nothing varies


def test_finalize_scores_matches_the_oracle():
    p, g = EO.sparse_maps(4, 34, 97, seed=2)
    s = EO.map_sums(p, g)
    got = finalize_scores(torch.from_numpy(s), 34, 97)
    want = EO.scores(p, g)
    for k in ("mse", "rmse", "cosine", "spectral_angle", "xic_corr"):
        np.testing.assert_allclose(got[k], want[k], rtol=1e-12, atol=1e-12, err_msg=k)
    zero = finalize_scores(torch.zeros(1, 9, dtype=torch.float64), 2, 2)
    assert zero["cosine"][0] == 0 and zero["xic_corr"][0] == 0 and math.isfinite(zero["spectral_angle"][0])
