"""Float64 numpy restatement of the validation map scores (`dq_map_scores` + `finalize_scores`), written from the
definitions rather than from the kernel's shifted one-pass sums: centred column statistics, `np.ptp` for "constant"."""
import numpy as np


def map_sums(pred, truth):
    """(b, rt, mz) maps -> (b, 9) float64: sse, sum pg, sum p^2, sum g^2, sum_mz PG, sum P^2, sum G^2 (P, G: RT sums),
    sum_mz w r, sum_mz w (r: Pearson correlation of a column over RT, w = G; w = 0 for a constant truth column, r = 0
    for a constant predicted column)."""
    p = np.asarray(pred, dtype=np.float64)
    g = np.asarray(truth, dtype=np.float64)
    out = np.zeros((p.shape[0], 9))
    out[:, 0] = ((p - g) ** 2).sum((1, 2))
    out[:, 1] = (p * g).sum((1, 2))
    out[:, 2] = (p * p).sum((1, 2))
    out[:, 3] = (g * g).sum((1, 2))
    P, G = p.sum(1), g.sum(1)
    out[:, 4] = (P * G).sum(1)
    out[:, 5] = (P * P).sum(1)
    out[:, 6] = (G * G).sum(1)
    pc = p - p.mean(1, keepdims=True)
    gc = g - g.mean(1, keepdims=True)
    g_var = np.ptp(g, axis=1) > 0
    p_var = np.ptp(p, axis=1) > 0
    with np.errstate(divide="ignore", invalid="ignore"):
        r = (pc * gc).sum(1) / np.sqrt((pc * pc).sum(1) * (gc * gc).sum(1))
    r = np.where(g_var & p_var, np.clip(r, -1.0, 1.0), 0.0)
    w = np.where(g_var, G, 0.0)
    out[:, 7] = (w * r).sum(1)
    out[:, 8] = w.sum(1)
    return out


def scores(pred, truth):
    """Per-window {mse, rmse, cosine, spectral_angle, xic_corr} straight from the maps, float64."""
    p = np.asarray(pred, dtype=np.float64)
    g = np.asarray(truth, dtype=np.float64)
    b = p.shape[0]
    mse = ((p - g) ** 2).reshape(b, -1).mean(1)

    def cos(a, c):
        a, c = a.reshape(b, -1), c.reshape(b, -1)
        den = np.linalg.norm(a, axis=1) * np.linalg.norm(c, axis=1)
        return np.where(den > 0, (a * c).sum(1) / np.where(den > 0, den, 1.0), 0.0)

    s = map_sums(p, g)
    xic = np.where(s[:, 8] > 0, s[:, 7] / np.where(s[:, 8] > 0, s[:, 8], 1.0), 0.0)
    return {"mse": mse, "rmse": np.sqrt(mse), "cosine": cos(p, g),
            "spectral_angle": 1.0 - 2.0 * np.arccos(np.clip(cos(p.sum(1), g.sum(1)), -1.0, 1.0)) / np.pi,
            "xic_corr": xic}


def sparse_maps(b, rt, mz, seed, density=0.3):
    """Random non-negative sparse (truth, prediction) pairs in [0, 1]-ish: most columns vary, all-zero columns of the
    truth are constant (skipped), and column 0 of the prediction is flat (r = 0) wherever the truth varies there."""
    rng = np.random.default_rng(seed)
    g = rng.random((b, rt, mz)) * (rng.random((b, rt, mz)) < density)
    p = np.clip(g + 0.2 * rng.standard_normal((b, rt, mz)) * (rng.random((b, rt, mz)) < 0.5), 0.0, None)
    g[:, :, 1] = 0.25           # a constant, non-zero truth column
    p[:, :, 0] = 0.5            # a flat predicted column
    g[:, 0, 0], g[:, 1, 0] = 0.0, 1.0
    return p.astype(np.float32), g.astype(np.float32)
