"""GPU: the weight EMA — the fused dq_adamw_ema kernel against dq_adamw and a float64 evaluation, dq_swap, training with
the EMA on (unchanged parameters, the EMA recurrence, the sharded layout), `ema_weights()` for forward passes and
sampling, and the EMA in checkpoints (save, resume, checkpoints without it)."""
import copy
import math
import os
import random

import pytest
import torch

from _util import TINY, make_net

pytestmark = pytest.mark.gpu

LR, B1, B2, EPS, WD = 1e-3, 0.9, 0.999, 1e-8, 0.01


def _adamw_scalars(step):
    return LR, B1, B2, EPS, WD, LR / (1 - B1 ** step), math.sqrt(1 - B2 ** step)


def _placed(srcs, off):
    """Copies of `srcs` at element offset `off` of fresh buffers: offset 0 takes the 16-byte vector kernels, offset 1
    the scalar ones."""
    out = []
    for s in srcs:
        buf = torch.empty(s.numel() + 4, dtype=s.dtype, device=s.device)
        out.append(buf[off:off + s.numel()])
        out[-1].copy_(s)
    return out


def _kernel_inputs(n, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    sign = torch.where(torch.rand(n, device="cuda", generator=g) < 0.5, -1.0, 1.0)
    # weights bounded away from 0 and an EMA close to them: ema + w (p - ema) has no cancellation, so the one rounding
    # of p - ema cannot be amplified past the result's ulp
    p = sign * (0.01 + 0.05 * torch.rand(n, device="cuda", generator=g))
    grad = 0.01 * torch.randn(n, device="cuda", generator=g)
    m = 1e-3 * torch.randn(n, device="cuda", generator=g)
    v = 1e-5 * torch.rand(n, device="cuda", generator=g)
    ema = p * (1 + 1e-2 * torch.randn(n, device="cuda", generator=g))
    return p, grad, m, v, ema


def _ulp(x):
    a = x.abs()
    return (torch.nextafter(a, torch.full_like(a, math.inf)) - a).double()


@pytest.mark.parametrize("n", [1 << 20, 1000003, 7])
@pytest.mark.parametrize("ema_w", [0.9, 1.0 - 0.999])
def test_adamw_ema_matches_adamw_and_float64_ema(n, ema_w):
    """p, m, v bit-identical to dq_adamw on the vector and the scalar path (n % 4 != 0 included); the EMA of both paths
    bit-identical and within 1 ulp of ema + ema_w (p_new - ema) evaluated in float64."""
    from dquartic import _native as N

    src = _kernel_inputs(n, seed=n % 97)
    coef = torch.tensor([0.0, 0.75], device="cuda")   # clip coefficient != 1
    w32 = float(torch.tensor(ema_w, dtype=torch.float32))
    emas = []
    for off in (0, 1):
        p, g, m, v = _placed(src[:4], off)
        p2, g2, m2, v2, e2 = _placed(src, off)
        N.call("dq_adamw", p, g, m, v, n, coef, *_adamw_scalars(3))
        N.call("dq_adamw_ema", p2, g2, m2, v2, e2, n, coef, *_adamw_scalars(3), ema_w)
        assert torch.equal(p, p2) and torch.equal(m, m2) and torch.equal(v, v2), off
        assert torch.equal(g2, src[1])
        ref = src[4].double() + w32 * (p2.double() - src[4].double())
        assert bool(((e2.double() - ref).abs() <= _ulp(e2)).all()), off
        emas.append(e2.clone())
    assert torch.equal(emas[0], emas[1])


@pytest.mark.parametrize("n", [1 << 20, 1000003, 3])
def test_swap_exchanges_exactly(n):
    from dquartic import _native as N

    a0 = torch.randn(n, device="cuda")
    b0 = torch.randn(n, device="cuda")
    for off in (0, 1):
        a, b = _placed((a0, b0), off)
        N.call("dq_swap", a, b, n)
        assert torch.equal(a, b0) and torch.equal(b, a0), off


def _inputs(b, rt, mz, seed, sparse=0.3):
    g = torch.Generator().manual_seed(seed)
    x0 = torch.rand(b, rt, mz, generator=g) * (torch.rand(b, rt, mz, generator=g) < sparse)
    c2 = 0.5 * x0 + 0.5 * torch.rand(b, rt, mz, generator=g) * (torch.rand(b, rt, mz, generator=g) < sparse)
    c1 = torch.rand(b, rt, generator=g)
    noise = torch.rand(b, rt, mz, generator=g)
    return x0.cuda(), c2.cuda(), c1.cuda(), noise.cuda()


def _ema_model(seed, ema_decay, lr=1e-3):
    from dquartic.model.model import DDIMDiffusionModel

    net, _ = make_net(seed=seed)
    d = DDIMDiffusionModel(net, device="cuda")
    d.ema_decay = ema_decay
    d._prepare_training(lr)
    return d


def test_training_with_ema_leaves_the_parameters_unchanged_and_follows_the_recurrence():
    """3 `_train_one_batch` steps (fixed t and noise) with ema_decay = 0.999, and a second optimizer WITHOUT the EMA on
    a copy of the network fed the same gradients (the backward accumulates with atomics, so two backward passes need
    not agree in the last bit): the flat parameters stay torch.equal, and the EMA follows the recurrence over the
    parameter snapshots, recomputed here in float64."""
    from dquartic.model.model_interface import FusedAdamW

    d = _ema_model(seed=11, ema_decay=0.999)
    net, opt = d.model, d.optimizer
    twin = copy.deepcopy(net)
    twin_opt = FusedAdamW(twin, lr=opt.param_groups[0]["lr"])
    n = net.n_trainable_flat
    real_step = opt.step

    def step(**kw):
        twin.flat_grads()[:n].copy_(net.flat_grads()[:n])
        twin_opt.step(**kw)
        real_step(**kw)

    opt.step = step
    ref = net.flat_params()[:n].double().clone()
    x0, c2, c1, noise = _inputs(2, 6, 320, 5)
    t = torch.tensor([30, 700], device="cuda")
    for k in range(3):
        d._train_one_batch(x0, ms2_cond=c2, ms1_cond=c1, noise=noise, t=t)
        p = net.flat_params()[:n]
        assert torch.equal(p, twin.flat_params()[:n]), k
        w = float(torch.tensor(1.0 - min(0.999, (1 + k) / (10 + k)), dtype=torch.float32))
        ref = ref + w * (p.double() - ref)
        err = float((opt._ema.double() - ref).abs().max() / ref.abs().max())
        assert err < 1e-6, (k, err)
    assert opt.ema_updates == 3 and twin_opt._ema is None
    assert not torch.equal(opt._ema, net.flat_params()[:n])


def test_sharded_ema_layout_matches_unsharded(monkeypatch):
    """set_sharding(rank, 2, ranges) for rank 0 and rank 1 in turn, fixed gradients, no clipping (no all-reduce), the
    parameter all-gather replaced by a recorder: every EMA segment of a rank is bit-identical to the unsharded EMA at
    the same flat offsets.  Per rank, too: swap_ema() exchanges exactly this rank's segments (and issues one gather per
    sharded range), a second swap restores the parameters and the EMA bit for bit, and load_ema_state_dict() of the
    unsharded EMA puts this rank's pieces at its state offsets."""
    from dquartic.model.model_interface import FusedAdamW

    gathered = []

    class _Done:
        def wait(self):
            pass

    def fake_all_gather(out, inp, async_op=False, **kw):
        gathered.append((out.numel(), inp.numel()))
        return _Done()

    monkeypatch.setattr(torch.distributed, "all_gather_into_tensor", fake_all_gather)
    base, _ = make_net(seed=12)
    n = base.n_trainable_flat
    ranges = sorted((o, c) for o, c in base.early_grad_ranges() if c % 2 == 0)
    keep = torch.zeros(n, device="cuda")    # no gradient in the alignment padding, as in training
    for name, par in base._params.items():
        if par.requires_grad:
            base._view(keep, name).fill_(1.0)
    grads = [1e-2 * keep * torch.randn(n, device="cuda", generator=torch.Generator(device="cuda").manual_seed(k))
             for k in range(3)]

    def run(rank):
        net = copy.deepcopy(base)
        opt = FusedAdamW(net, lr=1e-3, ema_decay=0.9)
        if rank is not None:
            opt.set_sharding(rank, 2, ranges)
        for gk in grads:
            net.flat_grads()[:n].copy_(gk)
            opt.step(max_grad_norm=None)
        return opt

    full = run(None)
    assert not gathered
    for rank in (0, 1):
        opt = run(rank)
        assert gathered == [(c, c // 2) for _ in grads for _, c in ranges]
        gathered.clear()
        assert opt._ema.numel() < n
        for (o, cnt, so) in opt._segments:
            assert torch.equal(opt._ema[so:so + cnt], full._ema[o:o + cnt]), (rank, o)
            assert torch.equal(opt._m[so:so + cnt], full._m[o:o + cnt]), (rank, o)
        p = opt.net.flat_params()
        live, ema = p.clone(), opt._ema.clone()
        opt.swap_ema()
        assert gathered == [(c, c // 2) for _, c in ranges]
        gathered.clear()
        swapped = live.clone()
        for (o, cnt, so) in opt._segments:
            swapped[o:o + cnt] = ema[so:so + cnt]
            assert torch.equal(opt._ema[so:so + cnt], live[o:o + cnt]), (rank, o)
        assert torch.equal(p, swapped)            # this rank's segments exchanged, the rest untouched
        opt.swap_ema()
        gathered.clear()
        assert torch.equal(p, live) and torch.equal(opt._ema, ema)
        fresh = FusedAdamW(copy.deepcopy(base), lr=1e-3, ema_decay=0.9)
        fresh.set_sharding(rank, 2, ranges)
        fresh.load_ema_state_dict(full.ema_state_dict(), full.ema_updates)
        assert fresh.ema_updates == 3 and torch.equal(fresh._ema, opt._ema)


def test_ema_weights_context_forward_sampling_and_restore(tmp_path):
    from dquartic.model.unet1d import UNet1d

    d = _ema_model(seed=13, ema_decay=0.9)
    net, opt = d.model, d.optimizer
    x0, c2, c1, noise = _inputs(4, 6, 320, 7)
    for _ in range(3):
        d._train_one_batch(x0, ms2_cond=c2, ms1_cond=c1)
    sd_ema = opt.ema_state_dict()
    assert list(sd_ema) == list(net.state_dict()) and len(sd_ema) == 396
    fresh = UNet1d(dim=TINY["dim"], channels=1, dim_mults=tuple(TINY["dim_mults"]), conditional=True,
                   init_cond_channels=1, attn_cond_channels=1, downsample_dim=TINY["downsample_dim"]).cuda()
    fresh.load_state_dict(sd_ema)
    fresh.eval()
    net.eval()
    t = torch.tensor([10, 200, 500, 900], device="cuda")
    n_c2, n_c1 = d.normalize(c2), d.normalize(c1)
    p_before = net.flat_params().clone()
    with torch.no_grad():
        out_before = net(noise, t, n_c2, n_c1).clone()
        out_fresh = fresh(noise, t, n_c2, n_c1)
    assert not torch.equal(out_before, out_fresh)

    def cond_fn(ids):
        idx = torch.tensor(ids, device="cuda")
        return c2[idx], c1[idx]

    with d.ema_weights() as m:
        assert m is net
        sd_in = net.state_dict()
        assert all(torch.equal(sd_in[k], v) for k, v in sd_ema.items())
        with torch.no_grad():
            assert torch.equal(net(noise, t, n_c2, n_c1), out_fresh)
        _, maps = d.sample_windows([0, 1, 2, 3], cond_fn, seed=3, num_steps=3, chunk=2, rank=0, world=1,
                                   cuda_graph=True)
        with pytest.raises(RuntimeError):
            opt.step()
        with pytest.raises(RuntimeError):      # would write the EMA as model_state_dict
            d.save_checkpoint(None, 0, 1.0, str(tmp_path / "inside.ckpt"))
    assert not os.path.exists(tmp_path / "inside.ckpt")
    assert torch.equal(net.flat_params(), p_before)
    with torch.no_grad():
        assert torch.equal(net(noise, t, n_c2, n_c1), out_before)   # the bf16 GEMM operands were recast back
    # the same windows sampled by the EMA-loaded fresh network
    from dquartic.model.model import DDIMDiffusionModel
    df = DDIMDiffusionModel(fresh, device="cuda")
    xT = torch.empty(4, 6, 320, device="cuda")
    for w in range(4):
        xT[w].normal_(generator=torch.Generator(device="cuda").manual_seed(d.window_seed(3, w)))
    with torch.no_grad():
        ref, _ = df.sample(xT, c2, c1, num_steps=3)
    assert torch.equal(maps, ref.cpu())
    # an exception inside the context still restores the live weights
    with pytest.raises(KeyError):
        with d.ema_weights():
            raise KeyError("boom")
    assert torch.equal(net.flat_params(), p_before)


def _tiny_loader(tmp_path):
    import numpy as np
    from dquartic.utils.data_loader import DeviceBatchLoader, DIAMSDataset
    from dquartic.utils.synthetic import synth_pool

    ms2, ms1 = synth_pool(12, 6, 320, seed=0)
    np.save(tmp_path / "ms2.npy", ms2)
    np.save(tmp_path / "ms1.npy", ms1)
    ds = DIAMSDataset(ms2_file=str(tmp_path / "ms2.npy"), ms1_file=str(tmp_path / "ms1.npy"), normalize="minmax")
    return DeviceBatchLoader(ds, 4, "cuda", pool="hbm", batches_per_epoch=3)


def _fixed_steps(d, n_steps):
    n = d.model.n_trainable_flat
    for k in range(n_steps):
        g = 1e-2 * torch.randn(n, device="cuda", generator=torch.Generator(device="cuda").manual_seed(100 + k))
        d.model.flat_grads()[:n].copy_(g)
        d.optimizer.step(max_grad_norm=d.max_grad_norm)


def test_checkpoints_carry_the_ema_and_resume_it_exactly(tmp_path, capsys):
    from dquartic.model.model import DDIMDiffusionModel
    from dquartic.model.unet1d import UNet1d

    loader = _tiny_loader(tmp_path)
    ckpt = str(tmp_path / "best.ckpt")
    net, _ = make_net(seed=1)
    d = DDIMDiffusionModel(net, device="cuda")
    d.ema_decay = 0.99
    random.seed(1)
    torch.manual_seed(1)
    d.train(loader, 4, 2, warmup_epochs=1, learning_rate=1e-4, use_wandb=False, checkpoint_path=ckpt)
    latest = str(tmp_path / "dquartic_latest_checkpoint.ckpt")
    ck = torch.load(latest, weights_only=False)
    assert set(ck) == {"epoch", "model_state_dict", "optimizer_state_dict", "scheduler_state_dict", "best_loss",
                       "ema_state_dict", "ema_updates"}
    assert ck["ema_updates"] == 6 and len(ck["ema_state_dict"]) == 396
    assert all(v.device.type == "cpu" for v in ck["ema_state_dict"].values())
    plain = UNet1d(dim=TINY["dim"], channels=1, dim_mults=tuple(TINY["dim_mults"]), conditional=True,
                   init_cond_channels=1, attn_cond_channels=1, downsample_dim=TINY["downsample_dim"])
    plain.load_state_dict(ck["ema_state_dict"])
    assert not torch.equal(ck["ema_state_dict"]["final_conv.weight"], ck["model_state_dict"]["final_conv.weight"])

    # resume into a fresh model: EMA and update count restored exactly
    d2 = DDIMDiffusionModel(make_net(seed=2)[0], device="cuda")
    d2.ema_decay = 0.99
    d2._prepare_training(1e-4)
    d2.load_checkpoint(None, latest, "cuda")
    assert d2.optimizer.ema_updates == 6
    got = d2.optimizer.ema_state_dict(device="cpu")
    assert all(torch.equal(got[k], v) for k, v in ck["ema_state_dict"].items())
    # N more steps of fixed gradients: resumed == uninterrupted, bit for bit
    _fixed_steps(d, 3)
    _fixed_steps(d2, 3)
    assert torch.equal(d2.optimizer._ema, d.optimizer._ema) and d2.optimizer.ema_updates == 9
    assert torch.equal(d2.model.flat_params(), d.model.flat_params())

    # with the EMA off the extra keys are ignored
    d3 = DDIMDiffusionModel(make_net(seed=3)[0], device="cuda")
    d3._prepare_training(1e-4)
    d3.load_checkpoint(None, latest, "cuda")
    assert d3.optimizer._ema is None
    d3.save_checkpoint(None, 0, 1.0, str(tmp_path / "no_ema.ckpt"))
    assert "ema_state_dict" not in torch.load(str(tmp_path / "no_ema.ckpt"), weights_only=False)

    # a checkpoint without the EMA, loaded with the EMA on: the EMA starts at the loaded weights
    capsys.readouterr()
    d4 = DDIMDiffusionModel(make_net(seed=4)[0], device="cuda")
    d4.ema_decay = 0.99
    d4._prepare_training(1e-4)
    _fixed_steps(d4, 2)
    d4.load_checkpoint(None, str(tmp_path / "no_ema.ckpt"), "cuda")
    assert "no weight EMA" in capsys.readouterr().out
    assert d4.optimizer.ema_updates == 0
    sd = d4.optimizer.ema_state_dict()
    live = d4.model.state_dict()
    assert all(torch.equal(sd[k], live[k]) for k in sd)
    assert all(torch.equal(sd[k].cpu(), v) for k, v in ck["model_state_dict"].items())
