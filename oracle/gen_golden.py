"""Golden-vector generator — TEST INFRASTRUCTURE, runs ONLY in the authoring container.

Imports the UNMODIFIED reference (`/root/reference/dquartic`) with the two shims under oracle/_shims
(rotary_embedding_torch, duckdb), runs it on CPU fp32 at batch 1 per sample (the only batch size the
reference supports) on deterministic inputs/weights, and writes small fixtures to tests/golden/.
The fixtures pin oracle/dquartic_oracle.py (tests/test_oracle_golden.py) and, through it and directly,
the CUDA path (tests/test_*_gpu.py).  /root/reference does not exist on the GPU box; nothing at test,
smoke or bench time reads it.

    python oracle/gen_golden.py            # regenerates tests/golden/*.npz
    DQUARTIC_REFERENCE=CHECKOUT python oracle/gen_golden.py   # from a checkout elsewhere (oracle/make_ref.py)
"""
import json
import os
import random
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(HERE, "_shims"))
sys.path.insert(0, "/root/reference")
if os.environ.get("DQUARTIC_REFERENCE"):
    sys.path.insert(0, os.environ["DQUARTIC_REFERENCE"])
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(ROOT, "diffusion-deconvolution-dia-msms-data_b200", "dquartic", "utils"))

import dquartic_oracle as O  # noqa: E402  (for det_params / shapes only — the numbers come from the reference)
from synthetic import synth_pool  # noqa: E402

from dquartic.model.unet1d import UNet1d  # noqa: E402  (reference)
from dquartic.model.model import DDIMDiffusionModel  # noqa: E402  (reference)
from dquartic.utils.data_loader import DIAMSDataset  # noqa: E402  (reference)

GOLD = os.path.join(ROOT, "tests", "golden")
os.makedirs(GOLD, exist_ok=True)
torch.set_num_threads(8)

TINY = dict(dim=4, channels=1, dim_mults=[1, 2, 2, 3, 3, 4, 4], conditional=True, init_cond_channels=1,
            attn_cond_channels=1, tfer_dim_mult=620, downsample_dim=320, simple=True)
DEFAULT = dict(TINY, downsample_dim=40000)
NOTEBOOK = dict(DEFAULT, dim_mults=[1, 2, 2, 2, 4, 4, 4])


def ref_model(cfg, seed=0):
    m = UNet1d(**{**cfg, "dim_mults": tuple(cfg["dim_mults"])})
    P = O.det_params(cfg, seed)
    sd = m.state_dict()
    assert list(sd.keys()) == list(P.keys()) or set(sd.keys()) == set(P.keys()), (
        set(sd.keys()) ^ set(P.keys()))
    for k in sd:
        assert tuple(sd[k].shape) == tuple(P[k].shape), (k, sd[k].shape, P[k].shape)
    m.load_state_dict(P)
    return m, P


def inputs(b, rt, mz, seed):
    x0 = O.det_tensor("x0", (b, rt, mz), 1.0, seed).abs().clamp(max=3) / 3  # in [0,1], mostly small
    x0 = x0 * (O.det_tensor("x0mask", (b, rt, mz), 1.0, seed) > 1.0)  # sparse like MS2
    other = O.det_tensor("other", (b, rt, mz), 1.0, seed).abs().clamp(max=3) / 3
    other = other * (O.det_tensor("othermask", (b, rt, mz), 1.0, seed) > 1.0)
    ms2_cond = 0.5 * x0 + 0.5 * other
    ms1 = torch.sigmoid(O.det_tensor("ms1", (b, rt), 1.5, seed))
    return x0.contiguous(), ms2_cond.contiguous(), ms1.contiguous()


def gen_schedule():
    out = {}
    for kind in ("cosine", "linear"):
        d = DDIMDiffusionModel(model_class=torch.nn.Identity(), num_timesteps=1000, beta_schedule_type=kind,
                               device="cpu")
        out[f"{kind}_betas"] = d.betas.numpy()
        out[f"{kind}_alphas"] = d.alphas.numpy()
        out[f"{kind}_alpha_bars"] = d.alpha_bars.numpy()
    dx = DDIMDiffusionModel(model_class=torch.nn.Identity(), num_timesteps=1000, pred_type="x0", device="cpu")
    out["cosine_x0_loss_weight"] = dx.loss_weight.numpy()
    out["steps50"] = torch.linspace(999, 0, 50, dtype=torch.long).numpy()
    out["steps7"] = torch.linspace(999, 0, 7, dtype=torch.long).numpy()
    np.savez_compressed(os.path.join(GOLD, "schedule.npz"), **out)
    print("schedule ok", out["cosine_alpha_bars"][[0, 499, 998, 999]])


def gen_keys():
    info = {}
    for name, cfg in (("default", DEFAULT), ("notebook", NOTEBOOK), ("tiny", TINY)):
        with torch.device("meta"):
            m = UNet1d(**{**cfg, "dim_mults": tuple(cfg["dim_mults"])})
        sd = m.state_dict()
        info[name] = {
            "cfg": cfg,
            "keys": [[k, list(v.shape)] for k, v in sd.items()],
            "total": int(sum(p.numel() for p in m.parameters())),
            "trainable": int(sum(p.numel() for p in m.parameters() if p.requires_grad)),
        }
        print(name, info[name]["total"], info[name]["trainable"], len(info[name]["keys"]))
    with open(os.path.join(GOLD, "state_dict_keys.json"), "w") as f:
        json.dump(info, f)


def gen_unet():
    b, rt, mz = 2, 34, TINY["downsample_dim"]
    m, _ = ref_model(TINY)
    m.eval()
    x = O.det_tensor("unet_x", (b, rt, mz), 1.0)
    ic = O.det_tensor("unet_ic", (b, rt, mz), 1.0)
    ac = O.det_tensor("unet_ac", (b, rt), 1.0)
    time = torch.tensor([7, 801], dtype=torch.long)
    with torch.no_grad():
        out = torch.cat([m(x[i:i + 1], time[i:i + 1], ic[i:i + 1], ac[i:i + 1]) for i in range(b)], dim=0)
    np.savez_compressed(os.path.join(GOLD, "unet_tiny.npz"), x=x.numpy(), time=time.numpy(), init_cond=ic.numpy(),
                        attn_cond=ac.numpy(), out=out.numpy())
    print("unet ok", out.shape, float(out.abs().mean()))


def gen_train():
    b, rt, mz = 2, 34, TINY["downsample_dim"]
    m, P = ref_model(TINY)
    m.train()
    ddim = DDIMDiffusionModel(model_class=m, num_timesteps=1000, device="cpu")
    x0, c2, c1 = inputs(b, rt, mz, 1)
    ts, noises, losses, eps_list = [], [], [], []
    grads = {k: torch.zeros_like(p) for k, p in m.named_parameters() if p.requires_grad}
    for i in range(b):
        seed = 100 + i
        torch.manual_seed(seed)
        t = torch.randint(0, 1000, (1,)).long()
        noise = torch.randn_like(x0[i:i + 1])
        ts.append(t)
        noises.append(noise)
        torch.manual_seed(seed)  # the reference draws the same t and noise itself (model.py:344-346)
        m.zero_grad()
        loss = ddim.train_step(x0[i:i + 1], c2[i:i + 1], c1[i:i + 1])
        assert loss.shape == (1,)
        loss.backward()
        losses.append(loss.detach())
        for k, p in m.named_parameters():
            if p.requires_grad:
                grads[k] += p.grad / b
    t = torch.cat(ts)
    noise = torch.cat(noises)
    losses = torch.cat(losses)
    # one clip + one AdamW step on the averaged gradient (batched oracle, SURVEY.md §8c)
    lr = 1e-3
    opt = torch.optim.AdamW(m.parameters(), lr=lr)
    for k, p in m.named_parameters():
        if p.requires_grad:
            p.grad = grads[k].clone()
    total_norm = torch.nn.utils.clip_grad_norm_(m.parameters(), max_norm=10.0)
    opt.step()
    new = {k: v.detach().clone() for k, v in m.state_dict().items()}
    # a second case whose norm exceeds the clip threshold: scale grads x1e4
    out = dict(x0=x0.numpy(), ms2_cond=c2.numpy(), ms1_cond=c1.numpy(), t=t.numpy(), noise=noise.numpy(),
               loss_per_sample=losses.numpy(), loss=np.float32(losses.mean().item()),
               total_norm=np.float32(total_norm.item()), lr=np.float32(lr))
    for k in ("init_conv.weight", "downs.0.0.block1.proj.weight", "mid_block1.block1.proj.weight",
              "mid_attn.fn.fn.to_qv.weight", "ups.6.2.fn.fn.to_out.1.g", "final_conv.bias", "time_mlp.1.weight"):
        out["new:" + k] = new[k].numpy()
    np.savez_compressed(os.path.join(GOLD, "train_tiny.npz"), **out)
    # the gradients in a file of their own: one archive with everything would pass 1 MB
    np.savez_compressed(os.path.join(GOLD, "train_tiny_grads.npz"), **{"grad:" + k: g.numpy() for k, g in grads.items()})
    print("train ok", losses, float(total_norm))


def gen_sample():
    b, rt, mz = 2, 34, TINY["downsample_dim"]
    m, _ = ref_model(TINY)
    ddim = DDIMDiffusionModel(model_class=m, num_timesteps=1000, device="cpu")
    x0, c2, c1 = inputs(b, rt, mz, 2)
    x_T = O.det_tensor("x_T", (b, rt, mz), 1.0, 2)
    out = dict(x_T=x_T.numpy(), ms2_cond=c2.numpy(), ms1_cond=c1.numpy())
    m.eval()
    for steps in (1, 6, 50):
        xs, pn = [], []
        with torch.no_grad():
            for i in range(b):
                x, p = ddim.sample(x_T[i:i + 1].clone(), c2[i:i + 1], c1[i:i + 1], num_steps=steps)
                xs.append(x)
                pn.append(p)
        out[f"x_{steps}"] = torch.cat(xs).numpy()
        out[f"pred_noise_{steps}"] = torch.cat(pn).numpy()
    # a single p_sample at t>0 and t==0
    with torch.no_grad():
        xp, ep = ddim.p_sample(x_T[0:1], 500, O.normalize(c2[0:1]), O.normalize(c1[0:1]))
        xz, ez = ddim.p_sample(x_T[0:1], 0, O.normalize(c2[0:1]), O.normalize(c1[0:1]))
    out.update(p500_x=xp.numpy(), p500_eps=ep.numpy(), p0_x=xz.numpy(), p0_eps=ez.numpy())
    np.savez_compressed(os.path.join(GOLD, "sample_tiny.npz"), **out)
    print("sample ok", float(np.abs(out["x_50"]).mean()))


def gen_data():
    n, rt, mz = 24, 34, 96
    ms2, ms1 = synth_pool(n, rt, mz, seed=7, density=0.2)
    tmp = "/tmp/dq_golden_pool"
    os.makedirs(tmp, exist_ok=True)
    np.save(os.path.join(tmp, "ms2.npy"), ms2)
    np.save(os.path.join(tmp, "ms1.npy"), ms1)
    ds = DIAMSDataset(ms2_file=os.path.join(tmp, "ms2.npy"), ms1_file=os.path.join(tmp, "ms1.npy"),
                      normalize="minmax")
    random.seed(1234)
    items = [ds[0] for _ in range(6)]
    pairs_small = sorted(ds.used_pairs)
    out = dict(ms2_pool=ms2, ms1_pool=ms1)
    for j, it in enumerate(items):
        for nm, arr in zip(("ms2_1", "ms1_1", "ms2_2", "ms1_2"), it):
            out[f"item{j}:{nm}"] = arr.numpy()
        out[f"item{j}:mix"] = (it[0] * 0.5 + it[2] * 0.5).numpy()
    # the exact (idx_1, idx_2) sequence of the rejection loop for N=520, two epochs of 64 draws
    class _Fake:
        def __init__(self, n):
            self.n = n

        def __len__(self):
            return self.n

        def __getitem__(self, i):
            return np.zeros((1, 1), np.int32)

    seq = []
    ds2 = DIAMSDataset.__new__(DIAMSDataset)
    ds2.ms2_data = _Fake(520)
    ds2.ms1_data = _Fake(520)
    ds2.used_pairs = set()
    random.seed(1234)
    import dquartic.utils.data_loader as DL
    orig = DL.random.randint
    rec = []

    def spy(a, b):
        v = orig(a, b)
        rec.append(v)
        return v

    DL.random.randint = spy
    try:
        for epoch in range(2):
            ds2.reset_epoch()
            for _ in range(64):
                before = len(rec)
                ds2._get_npy_pair()
                seq.append(rec[-2:])
    finally:
        DL.random.randint = orig
    out["pairs520"] = np.array(seq, dtype=np.int64)
    # float32 pool variant (numpy keeps float32 arithmetic there)
    ms2f = (ms2.astype(np.float32) * 1.37).astype(np.float32)
    ms1f = (ms1.astype(np.float32) * 0.73).astype(np.float32)
    np.save(os.path.join(tmp, "ms2f.npy"), ms2f)
    np.save(os.path.join(tmp, "ms1f.npy"), ms1f)
    dsf = DIAMSDataset(ms2_file=os.path.join(tmp, "ms2f.npy"), ms1_file=os.path.join(tmp, "ms1f.npy"),
                       normalize="minmax")
    random.seed(99)
    it = dsf[0]
    (i1, i2), = [p for p in dsf.used_pairs]
    out["f32_pool_ms2"] = ms2f
    out["f32_pool_ms1"] = ms1f
    for nm, arr in zip(("ms2_1", "ms1_1", "ms2_2", "ms1_2"), it):
        out[f"f32item:{nm}"] = arr.numpy()
    np.savez_compressed(os.path.join(GOLD, "data.npz"), **out)
    print("data ok", out["pairs520"][:4].tolist(), pairs_small[:3])


def _curve_run(cfg, b, rt, mz, steps, lr, perturb=0.0):
    """One reference training trajectory (batched-oracle semantics on the REFERENCE modules).  `perturb` > 0
    multiplies every initial weight by (1 + perturb * N(0,1)): the control run that measures how far the
    REFERENCE ITSELF moves under an fp32-rounding-sized change of its inputs."""
    m, _ = ref_model(cfg, seed=3)
    if perturb > 0:
        gp = torch.Generator().manual_seed(99)
        with torch.no_grad():
            for p in m.parameters():
                if p.requires_grad:
                    p.mul_(1 + perturb * torch.randn(p.shape, generator=gp))
    m.train()
    ddim = DDIMDiffusionModel(model_class=m, num_timesteps=1000, device="cpu")
    ms2, ms1 = synth_pool(12, rt, mz, seed=11, density=0.3)
    opt = torch.optim.AdamW(m.parameters(), lr=lr)
    rng = random.Random(4321)
    used = set()
    g = torch.Generator().manual_seed(777)
    losses, pair_log, t_log = [], [], []
    for s in range(steps):
        if s % 20 == 0:
            used.clear()
        grads = None
        step_losses = []
        for i in range(b):
            i1, i2 = O.pair_draw(rng, 12, used)
            a, c1, c, _ = O.minmax_pair(ms2[i1], ms1[i1], ms2[i2], ms1[i2])
            x0 = torch.from_numpy(a)[None]
            ms1c = torch.from_numpy(c1)[None]
            cond = O.mix(torch.from_numpy(a), torch.from_numpy(c))[None]
            t = torch.randint(0, 1000, (1,), generator=g)
            noise = torch.randn(x0.shape, generator=g)
            pair_log.append((i1, i2))
            t_log.append(int(t))
            # inject: reference maps injected noise n -> 2n-1 (model.py:346); to keep bit-exact noise we patch
            # torch.randint/randn_like for the duration of the call instead.
            orig_ri, orig_rl = torch.randint, torch.randn_like
            torch.randint = lambda *a_, **k_: t.clone()
            torch.randn_like = lambda *a_, **k_: noise.clone()
            try:
                m.zero_grad()
                loss = ddim.train_step(x0, cond, ms1c)
            finally:
                torch.randint, torch.randn_like = orig_ri, orig_rl
            loss.backward()
            step_losses.append(float(loss))
            gi = [p.grad.clone() / b for p in m.parameters() if p.requires_grad]
            grads = gi if grads is None else [x + y for x, y in zip(grads, gi)]
        for p, gr in zip([p for p in m.parameters() if p.requires_grad], grads):
            p.grad = gr
        torch.nn.utils.clip_grad_norm_(m.parameters(), max_norm=10.0)
        opt.step()
        losses.append(float(np.mean(step_losses)))
        if s % 50 == 0:
            print("curve step", s, losses[-1], flush=True)
    return np.array(losses, np.float32), np.array(pair_log, np.int64), np.array(t_log, np.int64)


def gen_curve():
    """200 optimizer steps at a shrunken shape, batch 2: (i) at the reference's shipped learning rate 1e-5
    (dquartic_train_config.json:15), (ii) at 5e-4 where the loss falls from 1.3 to ~0.5, and for each a CONTROL
    trajectory of the unmodified reference with its initial weights perturbed by 1e-6 relative (a few fp32 ulps):
    the control bounds how closely ANY second implementation can be expected to follow the curve."""
    cfg = dict(TINY, downsample_dim=128)
    b, rt, mz, steps = 2, 6, 128, 200
    out = {}
    for tag, lr in (("cfg_lr", 1e-5), ("", 5e-4)):
        losses, pairs, ts = _curve_run(cfg, b, rt, mz, steps, lr)
        ctrl, _, _ = _curve_run(cfg, b, rt, mz, steps, lr, perturb=1e-6)
        sfx = "_" + tag if tag else ""
        out["losses" + sfx] = losses
        out["losses_ctrl" + sfx] = ctrl
        out["lr" + sfx] = np.float64(lr)
        print("curve", lr, losses[0], losses[-1], "ctrl max rel dev", float(np.max(np.abs(ctrl - losses) / losses)))
    np.savez_compressed(os.path.join(GOLD, "curve_tiny.npz"), pairs=pairs, t=ts,
                        cfg=json.dumps(cfg), shape=np.array([b, rt, mz, steps]), **out)


if __name__ == "__main__":
    which = sys.argv[1:] or ["schedule", "keys", "unet", "train", "sample", "data", "curve"]
    for w in which:
        globals()["gen_" + w]()
