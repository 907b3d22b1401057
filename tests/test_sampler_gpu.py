"""Few-step ODE samplers on the GPU: the fused dq_dpm_step kernel, `sample(..., sampler=...)` on an analytic Gaussian
problem, the window-sharded driver and `dquartic predict`."""
import json
import math

import numpy as np
import pytest
import torch

import _ode_oracle as ODE
from _util import TINY, make_net

pytestmark = pytest.mark.gpu

U = 2.0 ** -24   # fp32 unit roundoff


def _ab():
    import dquartic_oracle as O
    return O.schedule_tables(1000, "cosine")[2].numpy().astype(np.float64)


# ------------------------------------------------------------------------------------------ kernel
@pytest.mark.parametrize("tau", [999, 500])
@pytest.mark.parametrize("pred_x0", [0, 1])
@pytest.mark.parametrize("mode", ["first", "second", "last_eps", "last"])
@pytest.mark.parametrize("n,off", [(4096, 0), (4099, 0), (4097, 1)])
def test_dpm_step_matches_float64(tau, pred_x0, mode, n, off):
    from dquartic import _native as N

    ab = _ab()
    alpha, sigma = np.float32(math.sqrt(ab[tau])), np.float32(math.sqrt(1 - ab[tau]))
    g = torch.Generator(device="cuda").manual_seed(tau * 7 + n + pred_x0)
    D_true = torch.randn(n + off, device="cuda", generator=g)
    eps = torch.randn(n + off, device="cuda", generator=g)
    x = (float(alpha) * D_true + float(sigma) * eps)[off:]
    out = ((D_true if pred_x0 else eps) + 0.05 * torch.randn(n + off, device="cuda", generator=g))[off:]
    hist0 = torch.randn(n + off, device="cuda", generator=g)[off:]
    if mode == "first":
        hist0.fill_(float("nan"))            # w_prev == 0: d_hist must not be read
    c_x, c_d = np.float32(0.93), np.float32(0.21)
    w_cur, w_prev = (np.float32(1.4), np.float32(-0.4)) if mode == "second" else (np.float32(1), np.float32(0))
    last = 1 if mode.startswith("last") else 0
    hist = hist0.clone()
    xn = torch.full_like(x, 7.0)
    e_out = torch.full_like(x, 7.0) if mode == "last_eps" else None
    N.call("dq_dpm_step", x, out, hist, xn, e_out, float(alpha), float(sigma), pred_x0, float(c_x), float(c_d),
           float(w_cur), float(w_prev), last, n)
    torch.cuda.synchronize()

    f = lambda t: t.double().cpu().numpy()
    X, O_, H = f(x), f(out), f(hist0)
    a, s = float(alpha), float(sigma)
    D = O_ if pred_x0 else (X - s * O_) / a
    Dmag = np.abs(O_) if pred_x0 else (np.abs(X) + s * np.abs(O_)) / a     # running-error magnitude of D
    errD = 3 * U * Dmag
    if last:
        np.testing.assert_array_less(np.abs(f(xn) - D), errD + 1e-30)
        assert torch.equal(hist, hist0)                          # the last step leaves d_hist alone
        if e_out is not None:
            E = (X - a * D) / s if pred_x0 else O_
            Emag = (np.abs(X) + a * Dmag) / s if pred_x0 else 0 * X
            np.testing.assert_array_less(np.abs(f(e_out) - E), 4 * U * Emag + 1e-30)
        return
    hterm = float(w_prev) * H if w_prev else 0.0
    ref = float(c_x) * X + float(c_d) * (float(w_cur) * D + hterm)
    mag = abs(float(c_x)) * np.abs(X) + abs(float(c_d)) * (abs(float(w_cur)) * Dmag + abs(float(w_prev)) * np.abs(
        np.nan_to_num(H)) * (w_prev != 0))
    bound = 6 * U * mag + abs(float(c_d)) * abs(float(w_cur)) * errD
    np.testing.assert_array_less(np.abs(f(xn) - ref), bound + 1e-30)
    np.testing.assert_array_less(np.abs(f(hist) - D), errD + 1e-30)


# ------------------------------------------------------------------------------------------ sampler
class _GaussNet(torch.nn.Module):
    """Optimal denoiser of elementwise Gaussian data (tests/_ode_oracle.py:Gauss) as the diffusion model's network."""

    def __init__(self, g, ab, pred_type, shape):
        super().__init__()
        self.mu = torch.from_numpy(g.mu).cuda().view(shape)
        self.s2 = torch.from_numpy(g.s * g.s).cuda().view(shape)
        self.ab = torch.from_numpy(ab).cuda()
        self.pred_type = pred_type

    def forward(self, x, t, init_cond=None, attn_cond=None):
        a2 = self.ab[t].view(-1, 1, 1)
        a = a2.sqrt()
        D = self.mu + a * self.s2 * (x.double() - a * self.mu) / (a2 * self.s2 + 1 - a2)
        out = D if self.pred_type == "x0" else (x.double() - a * D) / (1 - a2).sqrt()
        return out.float()


@pytest.mark.parametrize("pred_type", ["eps", "x0"])
def test_sample_solves_the_gaussian_ode(pred_type):
    from dquartic import _native as N
    from dquartic.model.model import DDIMDiffusionModel

    ab = _ab()
    shape = (25, 40, 100)
    g = ODE.Gauss(int(np.prod(shape)), ab, seed=0)
    d = DDIMDiffusionModel(torch.nn.Identity(), device="cuda", pred_type=pred_type, auto_normalize=False)
    d.model = _GaussNet(g, ab, pred_type, shape)
    xT = torch.from_numpy(g.x_T).float().cuda().view(shape)
    rms, launches = {}, {}
    with torch.no_grad():
        for sampler, order in (("ddim", 1), ("dpm++2m", 2)):
            for n in (10, 20, 40):
                before = N.launches
                x, eps = d.sample(xT, num_steps=n, sampler=sampler)
                launches[sampler, n] = N.launches - before
                got = x.double().cpu().numpy().ravel()
                rms[order, n] = g.rms(got)
                ref = ODE.ode_sample(g.denoise, ab, xT.double().cpu().numpy().ravel(), n, order)
                assert float(np.sqrt(np.mean((got - ref) ** 2))) < 5e-4, (sampler, n)   # fp32 vs fp64
                assert eps.shape == x.shape and bool(torch.isfinite(eps).all())   # no ms2_cond: epsilon at tau = 0
        before = N.launches
        d.sample(xT, num_steps=20)
        ref_launches = N.launches - before
    assert rms[2, 20] <= 5e-3 and rms[2, 10] <= 1.5e-2
    assert 1.7 <= rms[1, 20] / rms[1, 40] <= 2.3
    assert rms[2, 20] / rms[2, 40] >= 3.5
    assert launches["ddim", 20] == launches["dpm++2m", 20] == ref_launches == 20


# ------------------------------------------------------------------------------------------ driver
def _cond(b, rt, mz, seed):
    g = torch.Generator().manual_seed(seed)
    c2 = torch.rand(b, rt, mz, generator=g) * (torch.rand(b, rt, mz, generator=g) < 0.3)
    return c2.cuda(), torch.rand(b, rt, generator=g).cuda()


def _derived_xT(d, seed, ids, rt, mz):
    xT = torch.empty(len(ids), rt, mz, device="cuda")
    for k, w in enumerate(ids):
        xT[k].normal_(generator=torch.Generator(device="cuda").manual_seed(d.window_seed(seed, w)))
    return xT


@pytest.mark.parametrize("pred_type", ["eps", "x0"])
def test_sample_windows_dpm_is_independent_of_sharding_and_graph(pred_type):
    from dquartic import _native as N
    from dquartic.model.model import DDIMDiffusionModel

    net, _ = make_net(seed=4)
    d = DDIMDiffusionModel(net, device="cuda", pred_type=pred_type)
    c2, c1 = _cond(8, 6, 320, 5)

    def cond_fn(ids):
        idx = torch.tensor(ids, device="cuda")
        return c2[idx], c1[idx]

    ids = list(range(8))
    kw = dict(seed=11, num_steps=4, sampler="dpm++2m")    # 4 steps: first, second and final-first order updates
    _, full = d.sample_windows(ids, cond_fn, chunk=8, rank=0, world=1, cuda_graph=False, **kw)
    full = full.clone()
    for world, chunk, graph in ((1, 4, True), (2, 4, False), (2, 2, True), (4, 2, False), (4, 1, True)):
        parts = []
        for r in range(world):
            _, maps = d.sample_windows(ids, cond_fn, chunk=chunk, rank=r, world=world, cuda_graph=graph, **kw)
            parts.append(maps.clone())
        assert torch.equal(torch.cat(parts), full), (world, chunk, graph)
    xT = _derived_xT(d, 11, ids, 6, 320)
    with torch.no_grad():
        before = N.launches
        ref, _ = d.sample(xT, c2, c1, num_steps=4, sampler="dpm++2m")
        n_dpm = N.launches - before
        before = N.launches
        d.sample(xT, c2, c1, num_steps=4)
        n_ref = N.launches - before
    assert torch.equal(ref.cpu(), full)
    assert n_dpm == n_ref                                 # one fused update per model call, like the reference
    _, ddim = d.sample_windows(ids, cond_fn, chunk=8, rank=0, world=1, seed=11, num_steps=4, sampler="ddim")
    assert not torch.equal(ddim, full)


def test_reference_sampler_stays_the_default():
    from dquartic.model.model import DDIMDiffusionModel

    net, _ = make_net(seed=2)
    d = DDIMDiffusionModel(net, device="cuda")
    c2, c1 = _cond(4, 6, 320, 9)
    xT = _derived_xT(d, 3, range(4), 6, 320)
    with torch.no_grad():
        x_def, pn_def = d.sample(xT, c2, c1, num_steps=3)
        x_ref, pn_ref = d.sample(xT, c2, c1, num_steps=3, sampler="reference")
        # the reference's loop spelled out: p_sample at linspace(T-1, 0, 3), then the un-normalise tail
        x = xT
        for t in (999, 499, 0):
            x, _ = d.p_sample(x, t, d.normalize(c2), d.normalize(c1))
        x_loop = (x + 1) * 0.5
    assert torch.equal(x_def, x_ref) and torch.equal(pn_def, pn_ref)
    assert torch.equal(x_def, x_loop)

    def cond_fn(ids):
        idx = torch.tensor(ids, device="cuda")
        return c2[idx], c1[idx]

    _, maps = d.sample_windows(range(4), cond_fn, seed=3, num_steps=3, chunk=2, rank=0, world=1)
    assert torch.equal(maps, x_def.cpu())


# ------------------------------------------------------------------------------------------ dquartic predict
def _train_ckpt(tmp_path, with_ema):
    from dquartic.model.model import DDIMDiffusionModel

    net, _ = make_net(seed=6)
    d = DDIMDiffusionModel(net, device="cuda")
    d.ema_decay = 0.5 if with_ema else None
    d._prepare_training(1e-4)
    for k in range(3):
        g = 1e-1 * torch.randn(net.n_trainable_flat, device="cuda", generator=torch.Generator(device="cuda").manual_seed(k))
        net.flat_grads()[:net.n_trainable_flat].copy_(g)
        d.optimizer.step(max_grad_norm=d.max_grad_norm)
    path = str(tmp_path / ("ema.ckpt" if with_ema else "plain.ckpt"))
    d.save_checkpoint(None, 0, 1.0, path)
    return path


def _config(tmp_path):
    from dquartic.utils.config_loader import default_train_config

    cfg = default_train_config()
    cfg["model"]["UNet1d"].update({k: TINY[k] for k in cfg["model"]["UNet1d"]})
    cfg["data"]["parquet_directory"] = None
    path = tmp_path / "cfg.json"
    path.write_text(json.dumps(cfg))
    return str(path)


def _pool(tmp_path):
    from dquartic.utils.synthetic import synth_pool

    ms2, ms1 = synth_pool(7, 6, 320, seed=3, density=0.2)
    ms2[4] = 17                                          # a zero-range window
    np.save(tmp_path / "ms2.npy", ms2)
    np.save(tmp_path / "ms1.npy", ms1)
    return ms2, ms1


def _expected(state_dict, ms2, ms1, sampler, num_steps, seed):
    """Per-window min-max -> sample_windows -> pred * (max - min) + min, written out independently of the CLI."""
    from dquartic.model.model import DDIMDiffusionModel

    net, _ = make_net(seed=0)
    net.load_state_dict(state_dict)
    d = DDIMDiffusionModel(net, device="cuda")

    def mm(a):
        a = a.astype(np.float64).reshape(a.shape[0], -1)
        mn = a.min(1, keepdims=True)
        rng = a.max(1, keepdims=True) - mn
        rng[rng == 0] = 1
        return (a - mn) / rng, mn[:, 0], rng[:, 0]

    c2, mn, rng = mm(ms2)
    c1 = mm(ms1)[0]
    c2 = torch.from_numpy(c2).float().view(ms2.shape).cuda()
    c1 = torch.from_numpy(c1).float().cuda()

    def cond_fn(ids):
        idx = torch.tensor(ids, device="cuda")
        return c2[idx], c1[idx]

    _, maps = d.sample_windows(range(ms2.shape[0]), cond_fn, seed=seed, num_steps=num_steps, chunk=3, rank=0,
                               world=1, sampler=sampler)
    out = maps.numpy().copy()
    out *= rng.astype(np.float32)[:, None, None]
    out += mn.astype(np.float32)[:, None, None]
    return out


def _run(args):
    from click.testing import CliRunner
    from dquartic import cli

    res = CliRunner().invoke(cli.cli, args)
    assert res.exit_code == 0, (res.output, res.exception)
    return res.output


def test_predict_cli_writes_the_composed_pipeline_bit_for_bit(tmp_path, monkeypatch):
    from dquartic import cli

    monkeypatch.setattr(cli, "PREDICT_SLICE_CHUNKS", 1)  # several slices per run
    cfg = _config(tmp_path)
    ms2, ms1 = _pool(tmp_path)
    ema_ck, plain_ck = _train_ckpt(tmp_path, True), _train_ckpt(tmp_path, False)
    ck = torch.load(ema_ck, weights_only=False)
    assert not torch.equal(ck["ema_state_dict"]["final_conv.weight"], ck["model_state_dict"]["final_conv.weight"])
    base = ["predict", "--ms2-data-path", str(tmp_path / "ms2.npy"), "--ms1-data-path", str(tmp_path / "ms1.npy"),
            "--num-steps", "5", "--seed", "4", "--chunk", "2"]
    runs = {}
    for name, ckpt, weights in (("auto", ema_ck, "auto"), ("model", ema_ck, "model"), ("ema", ema_ck, "ema"),
                                ("plain", plain_ck, "auto")):
        out = str(tmp_path / f"{name}.npy")
        text = _run(base + ["--checkpoint-path", ckpt, "--weights", weights, "--output", out, cfg])
        assert ("EMA" in text) == (name in ("auto", "ema")), text
        runs[name] = np.load(out)
        assert runs[name].dtype == np.float32 and runs[name].shape == ms2.shape
        assert np.isfinite(runs[name]).all()
    want_ema = _expected(ck["ema_state_dict"], ms2, ms1, "dpm++2m", 5, 4)
    want_model = _expected(ck["model_state_dict"], ms2, ms1, "dpm++2m", 5, 4)
    assert np.array_equal(runs["auto"], want_ema) and np.array_equal(runs["ema"], want_ema)
    assert np.array_equal(runs["model"], want_model)
    assert not np.array_equal(want_ema, want_model)
    plain = torch.load(plain_ck, weights_only=False)["model_state_dict"]
    assert np.array_equal(runs["plain"], _expected(plain, ms2, ms1, "dpm++2m", 5, 4))
    # the reference sampler through the same path
    out = str(tmp_path / "ref.npy")
    _run(base + ["--checkpoint-path", plain_ck, "--sampler", "reference", "--output", out, cfg])
    assert np.array_equal(np.load(out), _expected(plain, ms2, ms1, "reference", 5, 4))


def test_predict_ranks_one_after_another_equal_one_rank(tmp_path, monkeypatch):
    from dquartic import cli
    from dquartic.model.model import DDIMDiffusionModel

    monkeypatch.setattr(cli, "PREDICT_SLICE_CHUNKS", 1)
    ms2, ms1 = _pool(tmp_path)
    net, _ = make_net(seed=8)
    d = DDIMDiffusionModel(net, device="cuda")
    one, two = str(tmp_path / "one.npy"), str(tmp_path / "two.npy")
    cli.predict_to_file(d, ms2, ms1, one, rank=0, world=1, num_steps=4, seed=1, chunk=2)
    for r in range(2):
        cli.predict_to_file(d, ms2, ms1, two, rank=r, world=2, num_steps=4, seed=1, chunk=2)
    a, b = np.load(one), np.load(two)
    assert np.array_equal(a, b) and np.isfinite(a).all()                  # window 4 has a zero range
