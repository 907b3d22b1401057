"""Float64 restatement of the few-step ODE samplers ("ddim", "dpm++2m") and an analytic test problem.

The reference has no such sampler: this follows DPM-Solver++(2M), Lu et al. 2022, arXiv:2211.01095, Algorithm 2 (data
prediction, multistep), with the first and the final update first order, on the quadratic grid of
`dquartic.model.model.sampler_grid`.  It is written from the paper's formulas (x_{i+1} = sigma_{i+1}/sigma_i x_i -
alpha_{i+1} (e^{-h_i} - 1) D_i), not from the product's coefficient helper, so that the two can be compared.

Test problem: elementwise Gaussian data x0 ~ N(mu, s^2).  For x_t = alpha x0 + sigma eps the optimal data prediction is
E[x0 | x_t] = mu + alpha s^2 (x_t - alpha mu) / (alpha^2 s^2 + sigma^2), and the probability-flow ODE keeps
z = (x_t - alpha mu) / sqrt(alpha^2 s^2 + sigma^2) constant, so its exact solution is known in closed form.
"""
import math

import numpy as np


def sampler_grid(T, N):
    """N strictly decreasing integer timesteps from T-1 to 0: q_i = rint((T-1)(1 - i/(N-1))^2) raised where needed.
    Closed form of the product's backward pass tau_i = max(q_i, tau_{i+1} + 1): tau_i = max_{j >= i} (q_j + j) - i."""
    i = np.arange(N)
    q = np.rint((T - 1) * (1.0 - i / (N - 1)) ** 2)
    return [int(v) for v in np.maximum.accumulate((q + i)[::-1])[::-1] - i]


def ode_sample(denoise_fn, alpha_bars, x_T, N, order):
    """`denoise_fn(x, t) -> D` (the data prediction at integer timestep t).  Order 1 is DDIM with the true previous
    alpha_bar, order 2 DPM-Solver++(2M).  Returns D at t = 0, all in float64."""
    ab = np.asarray(alpha_bars, dtype=np.float64)
    taus = sampler_grid(len(ab), N)
    alpha = [math.sqrt(ab[t]) for t in taus]
    sigma = [math.sqrt(1.0 - ab[t]) for t in taus]
    lam = [math.log(a / s) for a, s in zip(alpha, sigma)]
    x = np.asarray(x_T, dtype=np.float64)
    d_prev = None
    for i in range(N - 1):
        d = denoise_fn(x, taus[i])
        h = lam[i + 1] - lam[i]
        if order == 2 and 0 < i < N - 2:
            r = (lam[i] - lam[i - 1]) / h
            dd = (1 + 1 / (2 * r)) * d - 1 / (2 * r) * d_prev
        else:
            dd = d
        x = sigma[i + 1] / sigma[i] * x - alpha[i + 1] * (math.exp(-h) - 1.0) * dd
        d_prev = d
    return denoise_fn(x, taus[-1])


def reference_chain(denoise_fn, alpha_bars, x_T, N):
    """The reference's sampler (linear grid, every step lands on alpha_bars[t-1]) with the same denoiser, in float64."""
    ab = np.asarray(alpha_bars, dtype=np.float64)
    x = np.asarray(x_T, dtype=np.float64)
    for t in np.linspace(len(ab) - 1, 0, N).astype(np.int64):   # torch.linspace(..., dtype=long) truncates alike
        t = int(t)
        d = denoise_fn(x, t)
        if t == 0:
            return d
        eps = (x - math.sqrt(ab[t]) * d) / math.sqrt(1.0 - ab[t])
        x = math.sqrt(ab[t - 1]) * d + math.sqrt(1.0 - ab[t - 1]) * eps
    return x


class Gauss:
    """Elementwise Gaussian data, mu ~ U(-1, 1), s ~ U(0.05, 0.5), and x_T ~ N(0, 1), from a fixed seed."""

    def __init__(self, n, alpha_bars, seed=0):
        rng = np.random.default_rng(seed)
        self.mu = rng.uniform(-1.0, 1.0, n)
        self.s = rng.uniform(0.05, 0.5, n)
        self.x_T = rng.standard_normal(n)
        self.ab = np.asarray(alpha_bars, dtype=np.float64)

    def denoise(self, x, t):
        a2 = self.ab[t]
        a = math.sqrt(a2)
        s2 = self.s * self.s
        return self.mu + a * s2 * (x - a * self.mu) / (a2 * s2 + (1.0 - a2))

    def exact(self):
        """D at t = 0 of the exact probability-flow ODE solution started from x_T at t = T-1."""
        T = len(self.ab)
        aT, a0 = math.sqrt(self.ab[T - 1]), math.sqrt(self.ab[0])
        s2 = self.s * self.s
        z = (self.x_T - aT * self.mu) / np.sqrt(self.ab[T - 1] * s2 + 1.0 - self.ab[T - 1])
        x0 = a0 * self.mu + z * np.sqrt(self.ab[0] * s2 + 1.0 - self.ab[0])
        return self.denoise(x0, 0)

    def rms(self, got):
        return float(np.sqrt(np.mean((np.asarray(got, dtype=np.float64) - self.exact()) ** 2)))
