"""Few-step ODE samplers ("ddim", "dpm++2m") on the host: time grid, step coefficients, accuracy of the float64
restatement on an analytic Gaussian problem, and `dquartic predict`'s argument checks.  No GPU needed."""
import json
import math

import numpy as np
import pytest
import torch

import _ode_oracle as ODE
import dquartic_oracle as O
from dquartic.model.model import DDIMDiffusionModel, ode_coefs, sampler_grid

AB = O.schedule_tables(1000, "cosine")[2].numpy()


@pytest.mark.parametrize("n", [2, 3, 10, 20, 50, 999, 1000])
def test_grid_is_strictly_decreasing_from_T_minus_1_to_0(n):
    tau = sampler_grid(1000, n)
    assert len(tau) == n and tau[0] == 999 and tau[-1] == 0
    assert all(a > b for a, b in zip(tau, tau[1:]))
    assert tau == ODE.sampler_grid(1000, n)


def test_grid_is_the_identity_at_N_equals_T():
    assert sampler_grid(1000, 1000) == list(range(999, -1, -1))
    assert sampler_grid(7, 7) == list(range(6, -1, -1))


@pytest.mark.parametrize("n", [1, 0, 1001])
def test_grid_rejects_bad_step_counts(n):
    with pytest.raises(ValueError):
        sampler_grid(1000, n)


def test_first_order_step_is_alpha_next_D_plus_sigma_next_eps():
    rng = np.random.default_rng(0)
    taus = sampler_grid(1000, 20)
    steps = ode_coefs(AB, taus, 1)
    ab = AB.astype(np.float64)
    x, d = rng.standard_normal(1000), rng.standard_normal(1000)
    for i, (alpha, sigma, c_x, c_d, w_cur, w_prev, last) in enumerate(steps[:-1]):
        assert (w_cur, w_prev, last) == (1.0, 0.0, 0)
        assert alpha == math.sqrt(ab[taus[i]]) and sigma == math.sqrt(1 - ab[taus[i]])
        eps = (x - alpha * d) / sigma
        a1, s1 = math.sqrt(ab[taus[i + 1]]), math.sqrt(1 - ab[taus[i + 1]])
        np.testing.assert_allclose(c_x * x + c_d * d, a1 * d + s1 * eps, rtol=0, atol=1e-12)
    assert steps[-1][6] == 1 and len(steps) == 20


def test_second_order_only_strictly_inside():
    steps = ode_coefs(AB, sampler_grid(1000, 10), 2)
    w_prev = [s[5] for s in steps]
    assert w_prev[0] == 0 and w_prev[-2] == 0 and w_prev[-1] == 0
    assert all(w < 0 for w in w_prev[1:-2])
    assert all(abs(s[4] + s[5] - 1) < 1e-12 for s in steps)


def _kernel_semantics_sample(g, n_steps, order, pred_x0):
    """The loop of DDIMDiffusionModel._ode_sample with dq_dpm_step's formulas, in float64."""
    taus = sampler_grid(1000, n_steps)
    x, hist = g.x_T.copy(), None
    for t, (alpha, sigma, c_x, c_d, w_cur, w_prev, last) in zip(taus, ode_coefs(AB, taus, order)):
        D0 = g.denoise(x, t)
        out = D0 if pred_x0 else (x - alpha * D0) / sigma
        D = out if pred_x0 else (x - sigma * out) / alpha
        if last:
            return D
        x = c_x * x + c_d * (w_cur * D + (w_prev * hist if w_prev else 0.0))
        hist = D


@pytest.mark.parametrize("order", [1, 2])
@pytest.mark.parametrize("pred_x0", [False, True])
def test_product_coefficients_reproduce_the_oracle(order, pred_x0):
    g = ODE.Gauss(20000, AB, seed=1)
    ref = ODE.ode_sample(g.denoise, AB, g.x_T, 12, order)
    got = _kernel_semantics_sample(g, 12, order, pred_x0)
    np.testing.assert_allclose(got, ref, rtol=0, atol=1e-9)


@pytest.fixture(scope="module")
def rms():
    g = ODE.Gauss(100000, AB, seed=0)
    r = {(o, n): g.rms(ODE.ode_sample(g.denoise, AB, g.x_T, n, o)) for o in (1, 2) for n in (10, 20, 40)}
    r["reference", 50] = g.rms(ODE.reference_chain(g.denoise, AB, g.x_T, 50))
    return r


def test_oracle_accuracy_on_the_gaussian_problem(rms):
    assert rms[2, 20] <= 5e-3
    assert rms[2, 10] <= 1.5e-2
    assert 1.7 <= rms[1, 20] / rms[1, 40] <= 2.3          # first order
    assert rms[2, 20] / rms[2, 40] >= 3.5                  # second order
    assert rms[2, 20] < rms[1, 40]


def test_reference_chain_does_not_solve_the_ode_at_50_steps(rms):
    # the reference's step lands on alpha_bars[t-1] whatever the stride: characterised, not a target
    assert rms["reference", 50] >= 0.5


def test_sample_rejects_unknown_sampler_and_bad_step_counts():
    d = DDIMDiffusionModel(torch.nn.Identity(), device="cpu")
    x = torch.zeros(1, 2, 4)
    with pytest.raises(ValueError, match="unknown sampler"):
        d.sample(x, sampler="euler")
    for n in (1, 1001):
        with pytest.raises(ValueError, match="num_steps"):
            d.sample(x, num_steps=n, sampler="dpm++2m")


# ------------------------------------------------------------------------------------------ dquartic predict
def _predict_args(tmp_path, ms2_shape=(3, 6, 320), ms1_shape=(3, 6), **extra):
    from dquartic.utils.config_loader import default_train_config

    cfg = default_train_config()
    cfg["model"]["UNet1d"]["downsample_dim"] = 320
    cfg["data"]["parquet_directory"] = None
    (tmp_path / "cfg.json").write_text(json.dumps(cfg))
    np.save(tmp_path / "ms2.npy", np.zeros(ms2_shape, dtype=np.int32))
    np.save(tmp_path / "ms1.npy", np.zeros(ms1_shape, dtype=np.float32))
    torch.save({"model_state_dict": {}}, tmp_path / "ck.ckpt")
    args = ["predict", "--checkpoint-path", str(tmp_path / "ck.ckpt"), "--ms2-data-path", str(tmp_path / "ms2.npy"),
            "--ms1-data-path", str(tmp_path / "ms1.npy"), "--output", str(tmp_path / "out.npy")]
    for k, v in extra.items():
        args += [f"--{k.replace('_', '-')}", str(v)]
    return args + [str(tmp_path / "cfg.json")]


@pytest.mark.parametrize("case,kw,msg", [
    ("n", dict(ms1_shape=(4, 6)), "3 MS2 windows but 4 MS1"),
    ("mz", dict(ms2_shape=(3, 6, 321)), "downsample_dim is 320"),
    ("rt", dict(ms1_shape=(3, 7)), "6 retention-time points, MS1 has 7"),
    ("rank", dict(ms1_shape=(3, 6, 1)), "expected MS2 (N, rt, mz) and MS1 (N, rt)"),
    ("steps", dict(num_steps=1), "num-steps"),
    ("steps_hi", dict(num_steps=1001), "num-steps"),
    ("sampler", dict(sampler="euler"), "euler"),
    ("ema", dict(weights="ema"), "has no ema_state_dict"),
])
def test_predict_validates_inputs_before_any_cuda_call(tmp_path, monkeypatch, case, kw, msg):
    from click.testing import CliRunner
    from dquartic import cli

    def no_cuda(*a, **k):
        raise AssertionError("CUDA touched before the inputs were validated")

    monkeypatch.setattr(torch.cuda, "is_available", no_cuda)
    monkeypatch.setattr(torch.cuda, "set_device", no_cuda)
    shapes = {k: kw.pop(k) for k in ("ms2_shape", "ms1_shape") if k in kw}
    res = CliRunner().invoke(cli.cli, _predict_args(tmp_path, **shapes, **kw))
    assert res.exit_code == 2, (res.output, res.exception)
    assert msg in res.output
    assert not (tmp_path / "out.npy").exists()
