"""Held-out validation: a split of the slice pool, fixed mixtures of held-out slices with their clean maps, the
timestep bands of the denoising loss and the map scores (`ModelInterface.validate`, `ModelInterface.score_samples`,
`dquartic evaluate`).

Each synthetic mixture 0.5 ms2_1 + 0.5 ms2_2 has its clean map ms2_1 as ground truth, so held-out mixtures give both a
denoising loss at fixed (timestep, noise) and an exact score for sampled maps.  Everything here is drawn from fixed
seeds: two checkpoints are compared on identical inputs (common random numbers)."""
import math
import random
from collections import Counter

import numpy as np
import torch

SCORE_KEYS = ("cosine", "rmse", "spectral_angle", "xic_corr")


def band_timesteps(num_timesteps, bands):
    """Centres of `bands` equal strata of [0, T): t_k = floor((2k + 1) T / (2K))."""
    T, K = int(num_timesteps), int(bands)
    return [(2 * k + 1) * T // (2 * K) for k in range(K)]


def hold_out(dataset, fraction):
    """Hold out the last ceil(fraction * N) slices of `dataset` in file order (parquet: the sorted staging order): they
    are never drawn for training (`dataset.n_train`; fraction 1 holds out the whole pool, for evaluation only).  Returns
    the held-out index range (lo, hi)."""
    n = len(dataset)
    if not 0.0 < float(fraction) <= 1.0:
        raise ValueError(f"validation fraction must be in (0, 1], got {fraction}")
    lo = n - math.ceil(round(float(fraction) * n, 6))   # 0.07 * 100 = 7.000000000000001 holds out 7, not 8
    if float(fraction) < 1.0:
        dataset.n_train = lo
    return lo, n


def count_pairs(dataset, lo, hi):
    """Distinct unordered pairs of slices in [lo, hi) that `DIAMSDataset.draw_pair`'s rule admits."""
    m = hi - lo
    total = m * (m - 1) // 2
    meta = getattr(dataset, "pair_meta", None)
    if meta is not None:   # rows with the same (slice index, isolation window) are never paired
        total -= sum(k * (k - 1) // 2 for k in Counter(meta[lo:hi]).values())
    return total


def validation_pairs(dataset, lo, hi, windows, seed):
    """`windows` fixed (idx_1, idx_2) pairs of held-out slices, drawn with a private random.Random(seed) and the rule of
    `DIAMSDataset.draw_pair` (distinct indices, the parquet metadata rule, no repeated pair).  Host only."""
    avail = count_pairs(dataset, lo, hi)
    if avail < windows:
        raise ValueError(f"the {hi - lo} held-out slices give {avail} distinct pairs, fewer than the {windows} "
                         "validation windows asked for: lower `windows` or raise `fraction`")
    rng = random.Random(int(seed))
    used = set()
    return [dataset.pair_from(rng, lo, hi, used) for _ in range(int(windows))]


class ValidationSet:
    """The fixed validation problem: mixtures `cond` (W, rt, mz) with clean maps `x0` and MS1 conditioning `m1` (W, rt),
    all on the device in [0, 1]; the band timesteps `bands`; the noise map of window w drawn from a CUDA generator seeded with
    `DDIMDiffusionModel.window_seed(seed, w)` (as `sample_windows` draws x_T), shared by every band and every epoch."""

    def __init__(self, loader, pairs, num_timesteps, bands=10, seed=0, every_n_epochs=1):
        from ..model.model import DDIMDiffusionModel

        self.pairs = [tuple(int(i) for i in p) for p in pairs]
        self.bands = band_timesteps(num_timesteps, bands)
        self.seed = int(seed)
        self.every_n_epochs = int(every_n_epochs)
        self.x0, self.m1, _, _, self.cond = loader.make_batch(self.pairs, want_cond=True)
        dev = self.x0.device
        self.noise = torch.empty_like(self.x0)
        for w in range(len(self.pairs)):
            g = torch.Generator(device=dev)
            g.manual_seed(DDIMDiffusionModel.window_seed(self.seed, w))
            self.noise[w].normal_(generator=g)

    @property
    def windows(self):
        return len(self.pairs)

    def due(self, epoch):
        """Validate after epoch `epoch` (counting from 0)?"""
        return (epoch + 1) % self.every_n_epochs == 0


def finalize_scores(sums, rt, mz):
    """Per-window scores from `ModelInterface.map_scores` sums (b, 9): mse, rmse, cosine, spectral_angle =
    1 - 2 acos(cos(P, G)) / pi of the RT-summed spectra, and xic_corr = the G-weighted mean Pearson correlation of the m/z
    columns over RT (0 when no truth column varies).  Returns float64 numpy arrays."""
    s = torch.as_tensor(sums).detach().to("cpu", torch.float64).numpy()
    with np.errstate(divide="ignore", invalid="ignore"):
        mse = s[:, 0] / (int(rt) * int(mz))
        den = np.sqrt(s[:, 2]) * np.sqrt(s[:, 3])
        cosine = np.where(den > 0, s[:, 1] / den, 0.0)
        den_pg = np.sqrt(s[:, 5]) * np.sqrt(s[:, 6])
        cos_pg = np.where(den_pg > 0, s[:, 4] / den_pg, 0.0)
        xic = np.where(s[:, 8] > 0, s[:, 7] / s[:, 8], 0.0)
    return {"mse": mse, "rmse": np.sqrt(mse), "cosine": cosine,
            "spectral_angle": 1.0 - 2.0 * np.arccos(np.clip(cos_pg, -1.0, 1.0)) / np.pi, "xic_corr": xic}


def check_section(sec, for_train):
    """Range checks of the config's "validation" section (train: 0 < fraction < 1; evaluate: 0 < fraction <= 1; windows,
    bands and every_n_epochs integers >= 1, seed >= 0).  Returns the section with the defaults filled in."""
    out = {"windows": 64, "bands": 10, "seed": 0, "every_n_epochs": 1, **sec}
    unknown = set(out) - {"fraction", "windows", "bands", "seed", "every_n_epochs"}
    if unknown:
        raise ValueError(f"unknown validation keys {sorted(unknown)}")
    f = out.get("fraction")
    if isinstance(f, bool) or not isinstance(f, (int, float)) or not (0.0 < f < 1.0 if for_train else 0.0 < f <= 1.0):
        raise ValueError(f"validation.fraction must be in (0, {'1)' if for_train else '1]'}, got {f!r}")
    for k, least in (("windows", 1), ("bands", 1), ("seed", 0), ("every_n_epochs", 1)):
        v = out[k]
        if isinstance(v, bool) or not isinstance(v, int) or v < least:
            raise ValueError(f"validation.{k} must be an integer >= {least}, got {v!r}")
    return out
