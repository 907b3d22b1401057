"""GPU: round-2 coverage — tightened configuration parity (rt = 34 rows through the bf16 mid stage, north_star
tolerances), the BASELINE configs[4] shape class (dim 8, RT = 136), the secondary modes (x0 prediction + SNR weight, the
defined SIC loss, Softplus head), the harness (train two epochs + resume, _mix_to_device, predict), the window-sharded
sampling driver, the fused evaluation metric, the one-pass init_conv backward, and the tcgen05 LinearAttention backward
against the mma.sync one."""
import copy
import os
import random

import numpy as np
import pytest
import torch

from _util import TINY, make_net, rel_err

pytestmark = pytest.mark.gpu


def _cos(a, b):
    a = a.detach().double().cpu().flatten()
    b = b.detach().double().cpu().flatten()
    return float(torch.dot(a, b) / (a.norm() * b.norm()).clamp_min(1e-300))


def _inputs(b, rt, mz, seed, sparse=0.3):
    g = torch.Generator().manual_seed(seed)
    x0 = torch.rand(b, rt, mz, generator=g) * (torch.rand(b, rt, mz, generator=g) < sparse)
    c2 = 0.5 * x0 + 0.5 * torch.rand(b, rt, mz, generator=g) * (torch.rand(b, rt, mz, generator=g) < sparse)
    c1 = torch.rand(b, rt, generator=g)
    noise = torch.randn(b, rt, mz, generator=g)
    return x0, c2, c1, noise


@pytest.mark.parametrize("cfg_over,rt,mz,b", [
    (dict(dim=8, downsample_dim=320), 34, 320, 2),                    # widened net at the real RT (68 GEMM rows)
    (dict(dim=4, dim_mults=[1, 2, 4], downsample_dim=1300), 34, 1300, 2),
    (dict(dim=8, downsample_dim=320), 136, 320, 1),                   # BASELINE configs[4]: 2x channels, 4x longer RT axis
])
def test_configs_train_step_vs_oracle_north_star_tolerances(cfg_over, rt, mz, b):
    """Loss and every parameter gradient against the oracle with autograd at north_star's tolerances: bf16 paths
    rel <= 2e-2 (of the tensor's largest entry), cosine >= 0.999."""
    import dquartic_oracle as O
    from dquartic.model.model import DDIMDiffusionModel

    cfg = dict(TINY, **cfg_over)
    net, P = make_net(cfg, seed=5)
    net.train()
    d = DDIMDiffusionModel(net, device="cuda")
    x0, c2, c1, noise = _inputs(b, rt, mz, 17)
    t = torch.tensor([40, 870][:b])
    Pg = {k: v.clone().requires_grad_(not k.endswith("freqs")) for k, v in P.items()}
    _, _, ab = O.schedule_tables(1000, "cosine")
    ref_loss, _ = O.train_loss(Pg, cfg, ab, x0, c2, c1, t, noise)
    ref_loss.backward()
    net.zero_grad()
    loss = d.train_step(x0.cuda(), c2.cuda(), c1.cuda(), noise=((noise + 1) * 0.5).cuda(), t=t.cuda())
    loss.mean().backward()
    assert abs(float(loss.mean()) - float(ref_loss)) < 2e-3 * float(ref_loss)
    worst = (0.0, None)
    for k, v in Pg.items():
        if k.endswith("freqs"):
            continue
        e = rel_err(net._params[k].grad, v.grad)
        if e > worst[0]:
            worst = (e, k)
        assert e < 2e-2, (k, e)
        if v.numel() > 64:
            assert _cos(net._params[k].grad, v.grad) > 0.999, k
    print("worst gradient tensor", worst)


def test_config4_shape_class_sampling_vs_oracle():
    """dim = 8, RT = 136: three DDIM steps against the oracle (cosine >= 0.999)."""
    import dquartic_oracle as O
    from dquartic.model.model import DDIMDiffusionModel

    cfg = dict(TINY, dim=8, downsample_dim=320)
    net, P = make_net(cfg, seed=6)
    net.eval()
    d = DDIMDiffusionModel(net, device="cuda")
    x0, c2, c1, noise = _inputs(1, 136, 320, 9)
    _, _, ab = O.schedule_tables(1000, "cosine")
    with torch.no_grad():
        x, pn = d.sample(noise.cuda(), c2.cuda(), c1.cuda(), num_steps=3)
        rx, rpn = O.ddim_sample(P, cfg, ab, noise, c2, c1, 3)
    assert _cos(x, rx) > 0.999 and _cos(pn, rpn) > 0.999


@pytest.mark.parametrize("pred_type,w,softplus", [("x0", 0.0, False), ("eps", 0.3, False), ("x0", 0.2, True)])
def test_secondary_modes_vs_oracle(pred_type, w, softplus):
    """pred_type x0 with SNR weighting, the SIC loss (defined in oracle/dquartic_oracle.py:sic_loss), Softplus head."""
    import dquartic_oracle as O
    from dquartic.model.model import DDIMDiffusionModel
    from dquartic.model.unet1d import UNet1d

    cfg = TINY
    P = O.det_params(cfg, 4)
    net = UNet1d(dim=4, channels=1, dim_mults=tuple(cfg["dim_mults"]), conditional=True, init_cond_channels=1,
                 attn_cond_channels=1, downsample_dim=320, pos_output_only=softplus)
    net.load_state_dict(P)
    net = net.cuda().train()
    assert isinstance(net.final_act, torch.nn.Softplus if softplus else torch.nn.Identity)
    d = DDIMDiffusionModel(net, device="cuda", pred_type=pred_type, ms1_loss_weight=w)
    x0, c2, c1, noise = _inputs(2, 6, 320, 31)
    t = torch.tensor([100, 640])
    Pg = {k: v.clone().requires_grad_(not k.endswith("freqs")) for k, v in P.items()}
    _, _, ab = O.schedule_tables(1000, "cosine")
    ref, _ = O.train_loss_modes(Pg, cfg, ab, x0, c2, c1, t, noise, pred_type=pred_type, ms1_loss_weight=w,
                                pos_output_only=softplus)
    ref.mean().backward()
    net.zero_grad()
    loss = d.train_step(x0.cuda(), c2.cuda(), c1.cuda(), noise=((noise + 1) * 0.5).cuda(), ms1_loss_weight=w, t=t.cuda())
    assert loss.shape == (2,)
    loss.mean().backward()
    assert rel_err(loss, ref) < 5e-3
    for k in ("final_conv.weight", "init_conv.weight", "downs.0.2.fn.fn.to_qkv.weight", "mid_block1.block1.proj.weight",
              "ups.6.0.block1.proj.weight", "time_mlp.1.weight"):
        assert rel_err(net._params[k].grad, Pg[k].grad) < 3e-2, k
        assert _cos(net._params[k].grad, Pg[k].grad) > 0.999, k
    if pred_type == "x0":   # fused x0-mode reverse step: bit-exact against the eager op order of the reference
        net.eval()
        with torch.no_grad():
            xt = noise.cuda()
            xp, eps = d.p_sample(xt, 500, d.normalize(c2.cuda()), d.normalize(c1.cuda()))
            out = net(xt, torch.full((2,), 500, device="cuda"), d.normalize(c2.cuda()), d.normalize(c1.cuda()))
            sa, s1m, sap, s1mp = (torch.tensor(v, dtype=torch.float32, device="cuda") for v in d._step_coefs(500))
            eps_ref = (xt - sa * out) / s1m
            xp_ref = sap * out + s1mp * eps_ref
        assert torch.equal(eps, eps_ref) and torch.equal(xp, xp_ref)
        with torch.no_grad():
            x_last, _ = d.p_sample(xt, 0, d.normalize(c2.cuda()), d.normalize(c1.cuda()))
            out0 = net(xt, torch.zeros(2, dtype=torch.long, device="cuda"), d.normalize(c2.cuda()), d.normalize(c1.cuda()))
        assert torch.equal(x_last, out0)


def test_initconv_one_pass_backward_matches_generic_path():
    """dq_initconv_bwd (one pass, no data gradient of the conditioning channel) against the generic k7 wgrad + dgrad +
    per-sample dot path on the same inputs."""
    from dquartic.model.model import DDIMDiffusionModel

    x0, c2, c1, noise = _inputs(3, 6, 320, 41)
    t = torch.tensor([5, 500, 990])
    grads = []
    for force in (False, True):
        net, _ = make_net(seed=8)
        net.train()
        net._force_generic_initconv = force
        d = DDIMDiffusionModel(net, device="cuda")
        net.zero_grad()
        d.train_step(x0.cuda(), c2.cuda(), c1.cuda(), noise=((noise + 1) * 0.5).cuda(), t=t.cuda()).mean().backward()
        grads.append({k: net._params[k].grad.clone() for k in
                      ("init_conv.weight", "init_conv.bias", "init_cond_proj.to_scale_shift.1.weight",
                       "init_cond_proj.to_scale_shift.1.bias", "time_mlp.1.weight")})
    for k in grads[0]:
        assert rel_err(grads[0][k], grads[1][k]) < 2e-4, k


def _tiny_files(tmp_path, n=12, rt=6, mz=320, seed=0):
    from dquartic.utils.synthetic import synth_pool
    ms2, ms1 = synth_pool(n, rt, mz, seed=seed)
    np.save(tmp_path / "ms2.npy", ms2)
    np.save(tmp_path / "ms1.npy", ms1)
    return str(tmp_path / "ms2.npy"), str(tmp_path / "ms1.npy"), ms2, ms1


def test_mix_to_device_bit_exact_and_train_two_epochs_then_resume(tmp_path, capsys):
    """ModelInterface.train (reference model_interface.py:348-450): two epochs, checkpoints in the reference format,
    then a second call resumes at the saved epoch; `_mix_to_device` against the reference's arithmetic (1073-1075)."""
    from dquartic.model.model import DDIMDiffusionModel
    from dquartic.utils.data_loader import DeviceBatchLoader, DIAMSDataset

    f2, f1, _, _ = _tiny_files(tmp_path)
    ds = DIAMSDataset(ms2_file=f2, ms1_file=f1, normalize="minmax")
    random.seed(0)
    a, a1, b_, b1 = (torch.stack(z) for z in zip(*[ds[0] for _ in range(4)]))
    net, _ = make_net(seed=1)
    d = DDIMDiffusionModel(net, device="cuda")
    x_0, ms1_cond, ms2_cond = d._mix_to_device(a, a1, b_, (0.5, 0.5))
    assert torch.equal(x_0.cpu(), a) and torch.equal(ms1_cond.cpu(), a1)
    assert torch.equal(ms2_cond.cpu(), a * 0.5 + b_ * 0.5)
    x_0, _, ms2_cond = d._mix_to_device(a, a1, b_, (0.25, 0.75))
    assert torch.equal(ms2_cond.cpu(), a * 0.25 + b_ * 0.75)

    loader = DeviceBatchLoader(ds, 4, "cuda", pool="hbm", batches_per_epoch=3)
    ckpt = str(tmp_path / "best.ckpt")
    random.seed(1)
    torch.manual_seed(1)
    d.train(loader, 4, 2, warmup_epochs=1, learning_rate=1e-4, use_wandb=False, checkpoint_path=ckpt)
    out = capsys.readouterr().out
    assert "Epoch=1" in out and "Epoch=2" in out
    latest = str(tmp_path / "dquartic_latest_checkpoint.ckpt")
    assert os.path.exists(ckpt) and os.path.exists(latest)
    ck = torch.load(latest, weights_only=False)
    assert set(ck) == {"epoch", "model_state_dict", "optimizer_state_dict", "scheduler_state_dict", "best_loss"}
    assert ck["epoch"] == 1 and len(ck["model_state_dict"]) == 396
    # resume: a fresh model picks the weights and the optimizer state up and runs epochs 1..2 only
    net2, _ = make_net(seed=2)
    d2 = DDIMDiffusionModel(net2, device="cuda")
    d2.train(loader, 4, 3, warmup_epochs=1, learning_rate=1e-4, use_wandb=False, checkpoint_path=ckpt)
    out = capsys.readouterr().out
    assert "Resumed from" in out and "Epoch=1," not in out and "Epoch=3" in out
    assert d2.optimizer._step == 6 + 6           # 6 steps restored from the checkpoint, epochs 1 and 2 (3 batches each) run
    # the default config's wandb branch must not kill the loop (advisor finding): plotting is skipped with a warning
    d2.log_single_prediction  # exists
    with pytest.raises((ImportError, NotImplementedError)):
        d2.log_single_prediction(0, 0.0, loader)


def test_predict_returns_reference_dicts_and_predict_batch_scores_every_window(tmp_path):
    from dquartic.model.model import DDIMDiffusionModel
    from dquartic.utils.data_loader import DeviceBatchLoader, DIAMSDataset

    f2, f1, _, _ = _tiny_files(tmp_path, n=8)
    ds = DIAMSDataset(ms2_file=f2, ms1_file=f1, normalize="minmax")
    net, _ = make_net(seed=3)
    d = DDIMDiffusionModel(net, device="cuda")
    random.seed(2)
    loader = DeviceBatchLoader(ds, 3, "cuda", pool="hbm", batches_per_epoch=2)
    preds = d.predict(loader, num_steps=2)
    assert len(preds) == 2
    for p in preds:
        assert set(p) == {"ms2_1", "ms1_1", "mixture", "pred"}
        assert p["ms2_1"].shape == (3, 6, 320) and p["mixture"].shape == (3, 6, 320) and p["ms1_1"].shape == (3, 6)
        assert p["pred"].shape == (6, 320)            # the reference keeps item [0] only (model_interface.py:1150)
    x0, c2, c1, noise = _inputs(4, 6, 320, 3)
    pred, pn, cos = d.predict_batch(noise.cuda(), c2.cuda(), c1.cuda(), num_steps=2, target=x0.cuda())
    assert pred.shape == (4, 6, 320) and cos.shape == (4,)
    ref = torch.nn.functional.cosine_similarity(pred.flatten(1).double(), x0.cuda().flatten(1).double(), dim=1)
    assert torch.allclose(cos.double(), ref, atol=1e-5)
    res = d.predict_windows(loader, num_steps=2)
    assert len(res) == 2 and res[0]["pred"].shape == (3, 6, 320) and res[0]["cosine"].shape == (3,)


def test_sample_windows_is_independent_of_the_sharding_and_matches_sample():
    """configs[3]: windows {0..7} sampled as 1 x 8, 2 x 4 and 4 x 2 (rank blocks, different chunk sizes, with and
    without the CUDA graph) give bit-identical maps; x_T comes from (seed, window id) only."""
    from dquartic.model.model import DDIMDiffusionModel

    net, _ = make_net(seed=4)
    d = DDIMDiffusionModel(net, device="cuda")
    x0, c2, c1, _ = _inputs(8, 6, 320, 51)
    c2d, c1d = c2.cuda(), c1.cuda()

    def cond_fn(ids):
        idx = torch.tensor(ids, device="cuda")
        return c2d[idx], c1d[idx]

    ids = list(range(8))
    _, full = d.sample_windows(ids, cond_fn, seed=11, num_steps=3, chunk=8, rank=0, world=1, cuda_graph=False)
    full = full.clone()
    for world, chunk, graph in ((2, 4, False), (4, 2, False), (2, 2, True), (1, 3, True)):
        parts = []
        for r in range(world):
            got_ids, maps = d.sample_windows(ids, cond_fn, seed=11, num_steps=3, chunk=chunk, rank=r, world=world,
                                             cuda_graph=graph)
            lo, hi = d.shard_windows(8, r, world)
            assert got_ids == ids[lo:hi]
            parts.append(maps.clone())
        assert torch.equal(torch.cat(parts), full), (world, chunk, graph)
    # the same thing through `sample` with the x_T the driver derives
    xT = torch.empty(8, 6, 320, device="cuda")
    for w in ids:
        g = torch.Generator(device="cuda")
        g.manual_seed(d.window_seed(11, w))
        xT[w].normal_(generator=g)
    with torch.no_grad():
        ref, _ = d.sample(xT, c2d, c1d, num_steps=3)
    assert torch.equal(ref.cpu(), full)
    _, other = d.sample_windows(ids, cond_fn, seed=12, num_steps=3, chunk=8, rank=0, world=1)
    assert not torch.equal(other, full)


@pytest.mark.parametrize("C,L,pre", [(4, 4500, "downs.1.2"), (8, 1300, "downs.2.2"), (12, 2049, "downs.5.2"),
                                     (16, 700, "ups.0.2")])
def test_tcgen05_linear_attention_backward_matches_mma_sync_kernel(C, L, pre, tmp_path):
    """The tcgen05 / TMEM backward (q path) against the mma.sync TF32 kernel it replaces, same inputs, and the pipeline
    must not have timed out (dq_la_tc_last_error)."""
    import subprocess
    import sys
    from dquartic import _native

    net, _ = make_net(seed=7)
    net._ensure_grads()
    g = torch.Generator().manual_seed(2)
    R = 10
    x = (torch.randn(R, C, L, generator=g) * 1.5).cuda()
    dres = torch.randn(R, C, L, generator=g).cuda()
    net._gflat.zero_()
    out, saved = net._la_fwd(pre, x, True)
    dx = net._la_bwd(pre, saved, dres)
    torch.cuda.synchronize()
    assert _native.la_tc_last_error() is None
    names = [k for k in net._params if k.startswith(pre + ".")]
    got = {k: net._params[k].grad.clone().cpu() for k in names}
    f_in, f_out = str(tmp_path / "la_ab_in.pt"), str(tmp_path / "la_ab_out.pt")
    torch.save({"x": x.cpu(), "dres": dres.cpu()}, f_in)
    code = (
        "import sys, torch\n"
        f"sys.path[:0] = {sys.path!r}\n"
        "from _util import make_net\n"
        "net, _ = make_net(seed=7); net._ensure_grads(); net._gflat.zero_()\n"
        f"d = torch.load({f_in!r})\n"
        f"out, saved = net._la_fwd({pre!r}, d['x'].cuda(), True); dx = net._la_bwd({pre!r}, saved, d['dres'].cuda())\n"
        f"torch.save({{'dx': dx.cpu(), **{{k: net._params[k].grad.cpu() for k in net._params if k.startswith({pre!r} + '.')}}}}, {f_out!r})\n")
    env = dict(os.environ, DQ_LA_TC="0")
    subprocess.run([sys.executable, "-c", code], check=True, env=env)
    ref = torch.load(f_out)
    assert rel_err(dx, ref["dx"]) < 5e-3
    for k in names:
        assert rel_err(got[k], ref[k]) < 5e-3, k


@pytest.mark.parametrize("j,Lh", [(0, 625), (1, 1250), (2, 320), (3, 100), (4, 2500), (5, 1284)])
def test_upsample_backward_one_pass_matches_three_pass_composition(j, Lh):
    """dq_upconv_bwd_fused (half-rate rows staged, pairs folded in registers) against dq_upsample2x + dq_conv_bwd_fused +
    dq_fold2x: backward of Upsample = nearest x2 + Conv1d k3 (reference unet1d.py:93-96) at every channel pair of the up
    path, with 16-byte aligned and unaligned rows, ragged last tiles, accumulation into dx and dx not needed."""
    net, _ = make_net(seed=3)
    net._ensure_grads()
    wname, bname = f"ups.{j}.3.1.weight", f"ups.{j}.3.1.bias"
    cout, cin, _ = net.specs[wname]
    R = 5
    g = torch.Generator(device="cuda").manual_seed(100 + j)
    x = torch.randn(R, cin, Lh, device="cuda", generator=g)
    du = torch.randn(R, cout, 2 * Lh, device="cuda", generator=g)
    base = torch.randn(R, cin, Lh, device="cuda", generator=g)
    res = []
    for unfused in (True, False):
        net._force_unfused_upconv = unfused
        net.zero_grad()
        dx = net._upconv_bwd(du, x, wname, bname, True, None, 1)
        dxa = net._upconv_bwd(du, x, wname, bname, True, base.clone(), 1)
        none = net._upconv_bwd(du, x, wname, bname, False, None, 1)
        assert none is None
        torch.cuda.synchronize()
        res.append((dx.clone(), dxa.clone(), net._gw(wname).clone(), net._gw(bname).clone()))
    for a, b, what in zip(res[0], res[1], ("dx", "dx accumulated", "dW", "db")):
        assert rel_err(b, a) < 2e-5, (what, rel_err(b, a))


@pytest.mark.parametrize("i,L", [(0, 1250), (1, 2500), (2, 640), (3, 200), (4, 5000), (5, 1284)])
def test_downsample_backward_one_pass_matches_reindexing_composition(i, L):
    """dq_downconv_bwd_fused (half-rate dy rows staged, k4 / stride-2 taps resolved in place) against dq_s2d + dq_down_w +
    dq_conv_bwd_fused + dq_d2s: backward of Downsample = Conv1d(k4, s2, p1) (reference unet1d.py:110) at every channel pair
    of the down path, aligned and unaligned rows, ragged last tiles, accumulation into dx and dx not needed."""
    net, _ = make_net(seed=4)
    net._ensure_grads()
    wname, bname = f"downs.{i}.3.weight", f"downs.{i}.3.bias"
    cout, cin, k = net.specs[wname]
    assert k == 4
    R = 5
    g = torch.Generator(device="cuda").manual_seed(200 + i)
    x = torch.randn(R, cin, L, device="cuda", generator=g)
    du = torch.randn(R, cout, L // 2, device="cuda", generator=g)
    base = torch.randn(R, cin, L, device="cuda", generator=g)
    res = []
    for unfused in (True, False):
        net._force_unfused_downconv = unfused
        net.zero_grad()
        dx = net._downconv_bwd(du, x, wname, bname, True, None, 1)
        dxa = net._downconv_bwd(du, x, wname, bname, True, base.clone(), 1)
        none = net._downconv_bwd(du, x, wname, bname, False, None, 1)
        assert none is None
        torch.cuda.synchronize()
        res.append((dx.clone(), dxa.clone(), net._gw(wname).clone(), net._gw(bname).clone()))
    for a, b, what in zip(res[0], res[1], ("dx", "dx accumulated", "dW", "db")):
        assert rel_err(b, a) < 2e-5, (what, rel_err(b, a))


@pytest.mark.parametrize("i,L", [(0, 1250), (1, 2500), (2, 640), (3, 256), (4, 5000), (5, 1284), (0, 40000)])
def test_downsample_forward_pipelined_kernel_vs_torch(i, L):
    """Downsample = Conv1d(k4, stride 2, pad 1) (reference unet1d.py:110) through the bulk-copy pipelined forward kernel
    (stride-2 mode) against torch's fp32 convolution: every channel pair of the down path, aligned / unaligned rows,
    ragged last tiles."""
    net, _ = make_net(seed=5)
    wname, bname = f"downs.{i}.3.weight", f"downs.{i}.3.bias"
    cout, cin, k = net.specs[wname]
    R = 3
    g = torch.Generator(device="cuda").manual_seed(300 + i)
    x = torch.randn(R, cin, L, device="cuda", generator=g)
    y, _ = net._conv_fwd(x, None, wname, bname, 4, 2, 1, 1, L // 2)
    ref = torch.nn.functional.conv1d(x, net._w(wname).view(cout, cin, k), net._w(bname), stride=2, padding=1)
    assert y.shape == ref.shape
    assert rel_err(y, ref) < 1e-5, rel_err(y, ref)


@pytest.mark.parametrize("L,rt", [(40000, 3), (1250, 2), (333, 4), (128, 1)])
def test_init_conv_forward_pipelined_kernel_vs_torch(L, rt):
    """init_conv = Conv1d(2 -> dim, k7, pad 3) over cat(ConditionalScaleShift(cond), x) (reference unet1d.py:1107-1117,
    677-678) through the pipelined forward kernel (k7 mode, the per-sample scale / shift applied to the staged rows at
    existing positions only) against torch's fp32 ops."""
    net, _ = make_net(seed=6)
    b = 2
    R = b * rt
    net._time_path_fwd(torch.tensor([3, 700], device="cuda"), b, False)
    g = torch.Generator(device="cuda").manual_seed(17)
    net._SS.copy_(torch.randn(net._SS.shape, device="cuda", generator=g) * 0.5)
    ico = net.ss_off["init_cond_proj.to_scale_shift.1"]
    cond = torch.randn(R, 1, L, device="cuda", generator=g)
    x = torch.randn(R, 1, L, device="cuda", generator=g)
    y, _ = net._conv_fwd(cond, x, "init_conv.weight", "init_conv.bias", 7, 1, 3, 1, L, in_ss=ico, rps=rt)
    cout = net.specs["init_conv.weight"][0]
    sc = net._SS[:, ico].repeat_interleave(rt).view(R, 1, 1) + 1.0
    sh = net._SS[:, ico + 1].repeat_interleave(rt).view(R, 1, 1)
    ref = torch.nn.functional.conv1d(torch.cat([cond * sc + sh, x], 1), net._w("init_conv.weight").view(cout, 2, 7),
                                     net._w("init_conv.bias"), padding=3)
    assert rel_err(y, ref) < 1e-5, rel_err(y, ref)


def _misaligned(t):
    """A contiguous copy of `t` whose base address is 4 bytes past a 16-byte boundary (kernels must leave their vector paths)."""
    flat = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    v = flat[1:].view(t.shape)
    v.copy_(t)
    assert v.is_contiguous() and v.data_ptr() % 16 == 4
    return v


def test_resampling_kernels_accept_tensors_that_are_not_16_byte_aligned():
    """One-pass Upsample / Downsample backward and the pipelined Downsample / init_conv forward on tensors whose base
    pointers are only 4-byte aligned (views into larger buffers): same results as on aligned copies."""
    net, _ = make_net(seed=9)
    net._ensure_grads()
    R, L = 3, 512
    g = torch.Generator(device="cuda").manual_seed(5)
    # Upsample backward (ups.2: 12 -> 12 channels in the default net)
    wn, bn = "ups.2.3.1.weight", "ups.2.3.1.bias"
    cout, cin, _ = net.specs[wn]
    x = torch.randn(R, cin, L // 2, device="cuda", generator=g)
    du = torch.randn(R, cout, L, device="cuda", generator=g)
    res = []
    for f in (lambda t: t, _misaligned):
        net.zero_grad()
        dx = net._upconv_bwd(f(du), f(x), wn, bn, True, None, 1)
        res.append((dx.clone(), net._gw(wn).clone(), net._gw(bn).clone()))
    for a, b in zip(*res):
        assert rel_err(b, a) < 1e-5
    # Downsample backward and forward (downs.2: 8 -> 8)
    wn, bn = "downs.2.3.weight", "downs.2.3.bias"
    cout, cin, _ = net.specs[wn]
    x = torch.randn(R, cin, L, device="cuda", generator=g)
    du = torch.randn(R, cout, L // 2, device="cuda", generator=g)
    res = []
    for f in (lambda t: t, _misaligned):
        net.zero_grad()
        dx = net._downconv_bwd(f(du), f(x), wn, bn, True, None, 1)
        y, _ = net._conv_fwd(f(x), None, wn, bn, 4, 2, 1, 1, L // 2)
        res.append((dx.clone(), net._gw(wn).clone(), net._gw(bn).clone(), y.clone()))
    for a, b in zip(*res):
        assert rel_err(b, a) < 1e-5
    # init_conv forward
    b_, rt = 1, 3
    net._time_path_fwd(torch.tensor([11], device="cuda"), b_, False)
    ico = net.ss_off["init_cond_proj.to_scale_shift.1"]
    cond = torch.randn(rt, 1, L, device="cuda", generator=g)
    xx = torch.randn(rt, 1, L, device="cuda", generator=g)
    ys = [net._conv_fwd(f(cond), f(xx), "init_conv.weight", "init_conv.bias", 7, 1, 3, 1, L, in_ss=ico, rps=rt)[0].clone()
          for f in (lambda t: t, _misaligned)]
    assert rel_err(ys[1], ys[0]) < 1e-6


@pytest.mark.parametrize("rows,cols", [(300, 514), (256, 10000), (10000, 128), (64, 64), (33, 65), (2, 2)])
def test_cast_transpose_matches_torch_bit_exactly(rows, cols):
    """dq_cast_transpose (bf16 operand refresh of the mid-stage weights after AdamW): both layouts equal torch's
    round-to-nearest-even casts bit for bit, through the packed 64 x 64 kernel (even shapes) and the 32 x 32 one."""
    from dquartic import _native as N
    g = torch.Generator(device="cuda").manual_seed(rows * 31 + cols)
    x = torch.randn(rows, cols, device="cuda", generator=g)
    out = torch.empty(rows, cols, dtype=torch.bfloat16, device="cuda")
    out_t = torch.empty(cols, rows, dtype=torch.bfloat16, device="cuda")
    N.call("dq_cast_transpose", x, out, out_t, rows, cols)
    assert torch.equal(out, x.bfloat16())
    assert torch.equal(out_t, x.t().contiguous().bfloat16())


@pytest.mark.parametrize("rows,cols,ld,shift", [(72, 10000, 80, 0), (72, 10000, 80, -1), (72, 10000, 80, 1), (2304, 256, 2304, 0),
                                                (70, 130, 72, 1), (33, 65, 40, 0), (64, 64, 64, -1)])
def test_transpose_bf16_with_row_shift_matches_torch(rows, cols, ld, shift):
    """dq_transpose_bf16: out[c][r] = in[r + shift][c] (zero outside), leading dimension ld - the activation transposes of
    the mid-stage weight-gradient GEMMs, through the packed 64 x 64 kernel (even shapes) and the 32 x 32 one."""
    from dquartic import _native as N
    g = torch.Generator(device="cuda").manual_seed(rows + cols + shift)
    x = torch.randn(rows, cols, device="cuda", generator=g).bfloat16()
    out = torch.full((cols, ld), 7.0, dtype=torch.bfloat16, device="cuda")
    N.call("dq_transpose_bf16", x, out, rows, cols, ld, shift)
    ref = torch.zeros(rows, cols, dtype=torch.bfloat16, device="cuda")
    lo, hi = max(0, -shift), min(rows, rows - shift)
    ref[lo:hi] = x[lo + shift:hi + shift]
    assert torch.equal(out[:, :rows], ref.t())
    assert bool((out[:, rows:] == 7.0).all())       # the padding columns of the destination are left alone


@pytest.mark.parametrize("N,act,with_ss,with_res", [(10000, 1, True, False), (10000, 1, False, True), (20000, 1, True, True),
                                                    (520, 0, False, False), (1002, 1, True, True)])
def test_rownorm_forward_vector_and_scalar_kernels_vs_torch(N, act, with_ss, with_res):
    """dq_rownorm_fwd (RMSNorm(10000) + per-sample scale/shift + SiLU + residual of the mid stage, reference
    unet1d.py:126-140, 260-266) against torch: the 16-byte vector kernel (N % 4 == 0; the row kept in registers for N <=
    10240, re-read above) and the scalar kernel (N = 1002), fp32 and bf16 outputs."""
    from dquartic import _native as N_
    b, rt = 3, 5
    M = b * rt
    gen = torch.Generator(device="cuda").manual_seed(N + act)
    u = torch.randn(M, N, device="cuda", generator=gen)
    g = torch.rand(N, device="cuda", generator=gen) + 0.5
    ssw = 2 * N + 6                       # scale | shift of this producer start at column 2 of a wider SS buffer
    SS = torch.randn(b, ssw, device="cuda", generator=gen) * 0.3
    res = torch.randn(M, N, device="cuda", generator=gen) if with_res else None
    of = torch.empty(M, N, device="cuda")
    ob = torch.empty(M, N, dtype=torch.bfloat16, device="cuda")
    inv = torch.empty(M, device="cuda")
    ssp = SS.data_ptr() + 8 if with_ss else None
    N_.call("dq_rownorm_fwd", u, 0, g, ssp, ssw, act, res, of, ob, 0, inv, b, rt, N)
    nrm = u.norm(dim=1, keepdim=True).clamp_min(1e-12)
    z = u / nrm * g * (N ** 0.5)
    if with_ss:
        sc = SS[:, 2:2 + N].repeat_interleave(rt, 0)
        sh = SS[:, 2 + N:2 + 2 * N].repeat_interleave(rt, 0)
        z = z * (sc + 1) + sh
    if act == 1:
        z = torch.nn.functional.silu(z)
    if with_res:
        z = z + res
    assert rel_err(of, z) < 2e-6
    assert rel_err(ob.float(), z.bfloat16().float()) < 1e-2 and float((ob.float() - z).abs().max()) < 0.05 * float(z.abs().max())
    assert rel_err(inv, (1.0 / nrm).flatten()) < 1e-6
