"""ORACLE — TEST INFRASTRUCTURE ONLY.  Not shipped, not on the product path.

A CPU restatement (torch fp32, functional, no nn.Module from the reference) of the dquartic hot
path: the MS1-conditioned DDIM denoiser training step and DDIM sampling loop.  Only `tests/`,
`__graft_entry__.smoke()` and `bench.py`'s cpu_baseline / `--impl reference` leg may import it,
and there only as the checker or the timed CPU baseline.

Parity status: PINNED against the reference itself.  `oracle/gen_golden.py` imports the unmodified
reference from /root/reference (with the rotary / duckdb shims in oracle/_shims) in the authoring
container, runs it at batch 1 per sample (the only batch size it supports, SURVEY.md finding 1)
and commits the input/output vectors to tests/golden/*.npz; tests/test_oracle_golden.py checks
every function here against those vectors.  The single un-pinned spot is the third-party
`rotary-embedding-torch` arithmetic (pinned ^0.8.4, not vendored): restated from its published
semantics in `rope()` below.

Batched semantics (the reference has none, SURVEY.md §8c): a batch is the vmap of the b=1
reference — row r of sample i uses sample i's time embedding; loss = mean over all elements;
gradients are those of that mean loss; one clip_grad_norm_(10) and one AdamW step per batch.

All file:line citations are relative to /root/reference/dquartic/.
"""
import math

import torch
import torch.nn.functional as F

HEADS = 4
DIM_HEAD = 32


# ----------------------------------------------------------------------------- schedule (a1)
def cosine_beta_schedule(T, s=0.008):
    """model/model.py:32-54 — fp64."""
    x = torch.linspace(0, T, T + 1, dtype=torch.float64)
    ac = torch.cos(((x / T) + s) / (1 + s) * math.pi * 0.5) ** 2
    ac = ac / ac[0]
    betas = 1 - (ac[1:] / ac[:-1])
    return torch.clip(betas, 0, 0.999)


def linear_beta_schedule(T, beta_start=0.0001, beta_end=0.02):
    """model/model.py:14-29."""
    return torch.linspace(beta_start, beta_end, T, dtype=torch.float64)


def schedule_tables(T=1000, kind="cosine"):
    """model/model.py:196-202: betas fp64 -> fp32, alphas = 1 - betas (fp32), alpha_bars = cumprod fp32."""
    betas = (linear_beta_schedule(T) if kind == "linear" else cosine_beta_schedule(T)).to(torch.float32)
    alphas = (1.0 - betas).to(torch.float32)
    alpha_bars = torch.cumprod(alphas, dim=0).to(torch.float32)
    return betas, alphas, alpha_bars


def loss_weight_table(alpha_bars, pred_type):
    """model/model.py:206-213."""
    snr = alpha_bars / (1 - alpha_bars)
    if pred_type == "eps":
        return torch.ones_like(snr)
    if pred_type == "x0":
        return snr
    raise ValueError(f"Unknown pred_type: {pred_type}")


# ----------------------------------------------------------------------------- elementwise (a2, a3)
def normalize(x):
    """model/model.py:99."""
    return x * 2 - 1


def unnormalize(x):
    """model/model.py:112."""
    return (x + 1) * 0.5


def q_sample(alpha_bars, x0, t, noise):
    """model/model.py:239-242."""
    a = torch.sqrt(alpha_bars[t])[:, None, None]
    s = torch.sqrt(1.0 - alpha_bars[t])[:, None, None]
    return a * x0 + s * noise


def ddim_update(alpha_bars, x_t, eps, t):
    """model/model.py:265-289, pred_type == 'eps', eta = 0.  Note alpha_bars[t-1] regardless of stride."""
    ab = alpha_bars[t]
    x0_pred = (x_t - torch.sqrt(1.0 - ab) * eps) / torch.sqrt(ab)
    if t > 0:
        abp = alpha_bars[t - 1]
        return torch.sqrt(abp) * x0_pred + torch.sqrt(1.0 - abp) * eps
    return x0_pred


def ddim_timesteps(T, num_steps):
    """model/model.py:313."""
    return torch.linspace(T - 1, 0, num_steps, dtype=torch.long)


# ----------------------------------------------------------------------------- denoiser blocks (a7)
def rmsnorm(x, g):
    """model/unet1d.py:140: F.normalize(x, dim=1) * g * sqrt(C); F.normalize eps = 1e-12."""
    n = torch.sqrt((x * x).sum(dim=1, keepdim=True)).clamp_min(1e-12)
    return x / n * g * (x.shape[1] ** 0.5)


def sinusoidal_pos_emb(time, dim, theta=10000):
    """model/unet1d.py:211-218."""
    half = dim // 2
    e = math.log(theta) / (half - 1)
    f = torch.exp(torch.arange(half, dtype=torch.float32) * -e)
    a = time[:, None].to(torch.float32) * f[None, :]
    return torch.cat((a.sin(), a.cos()), dim=-1)


def time_mlp(P, time, dim):
    """model/unet1d.py:958-960: SinusoidalPosEmb -> Linear -> GELU(erf) -> Linear."""
    e = sinusoidal_pos_emb(time, dim)
    e = F.linear(e, P["time_mlp.1.weight"], P["time_mlp.1.bias"])
    e = F.gelu(e)
    return F.linear(e, P["time_mlp.3.weight"], P["time_mlp.3.bias"])


def block(P, pre, x, scale_shift=None):
    """model/unet1d.py:248-268: conv k3 p1 -> RMSNorm -> x*(scale+1)+shift -> SiLU (dropout p=0)."""
    x = F.conv1d(x, P[pre + ".proj.weight"], P[pre + ".proj.bias"], padding=1)
    x = rmsnorm(x, P[pre + ".norm.g"])
    if scale_shift is not None:
        scale, shift = scale_shift
        x = x * (scale + 1) + shift
    return F.silu(x)


def resnet_block(P, pre, x, t_emb, rows_per_sample):
    """model/unet1d.py:302-323.  Batched semantics: the (b, 2C) scale/shift of sample i is applied to all
    `rows_per_sample` rows of that sample (rows_per_sample = 1 for the mid blocks)."""
    ss = F.linear(F.silu(t_emb), P[pre + ".mlp.1.weight"], P[pre + ".mlp.1.bias"])  # (b, 2C)
    ss = ss.repeat_interleave(rows_per_sample, dim=0)[:, :, None]
    scale, shift = ss.chunk(2, dim=1)
    h = block(P, pre + ".block1", x, (scale, shift))
    h = block(P, pre + ".block2", h)
    if (pre + ".res_conv.weight") in P:
        res = F.conv1d(x, P[pre + ".res_conv.weight"], P[pre + ".res_conv.bias"])
    else:
        res = x
    return h + res


def linear_attention(P, pre, x):
    """model/unet1d.py:473-496 wrapped as Residual(PreNorm(.)) (unet1d.py:1017, 64-79, 163-176).
    `pre` is e.g. 'downs.0.2'."""
    xn = rmsnorm(x, P[pre + ".fn.norm.g"])
    R, C, L = x.shape
    qkv = F.conv1d(xn, P[pre + ".fn.fn.to_qkv.weight"])
    q, k, v = qkv.chunk(3, dim=1)
    q = q.reshape(R, HEADS, DIM_HEAD, L)
    k = k.reshape(R, HEADS, DIM_HEAD, L)
    v = v.reshape(R, HEADS, DIM_HEAD, L)
    q = q.softmax(dim=-2) * (DIM_HEAD ** -0.5)
    k = k.softmax(dim=-1)
    context = torch.einsum("bhdn,bhen->bhde", k, v)
    out = torch.einsum("bhde,bhdn->bhen", context, q).reshape(R, HEADS * DIM_HEAD, L)
    out = F.conv1d(out, P[pre + ".fn.fn.to_out.0.weight"], P[pre + ".fn.fn.to_out.0.bias"])
    out = rmsnorm(out, P[pre + ".fn.fn.to_out.1.g"])
    return out + x


def rope(t, freqs):
    """Third-party rotary-embedding-torch ^0.8.4 `rotate_queries_or_keys` on (b, h, n, d), restated:
    positions 0..n-1, angles pos*freqs repeated pairwise, interleaved-pair rotation of the first
    2*len(freqs) features, the rest pass through.  Call sites: model/unet1d.py:560-561."""
    n = t.shape[-2]
    ang = torch.arange(n, dtype=torch.float32, device=t.device)[:, None] * freqs[None, :]  # (n, 8)
    ang = ang.repeat_interleave(2, dim=-1)  # (n, 16)
    rd = ang.shape[-1]
    tr, tp = t[..., :rd], t[..., rd:]
    x1 = tr[..., 0::2]
    x2 = tr[..., 1::2]
    rot = torch.stack((-x2, x1), dim=-1).reshape(tr.shape)
    tr = tr * ang.cos() + rot * ang.sin()
    return torch.cat((tr, tp), dim=-1)


def mid_attention(P, x, cond):
    """model/unet1d.py:552-567 + 428-443 (non-flash) wrapped in Residual(PreNorm) (1030-1042).
    x (b, Cm, rt); cond (b, 8, rt)."""
    b, Cm, n = x.shape
    xn = rmsnorm(x, P["mid_attn.fn.norm.g"])
    qv = F.conv1d(xn, P["mid_attn.fn.fn.to_qv.weight"])
    q, v = qv.chunk(2, dim=1)
    k = F.conv1d(cond, P["mid_attn.fn.fn.to_k.weight"])
    hd = lambda z: z.reshape(b, HEADS, DIM_HEAD, n).permute(0, 1, 3, 2)  # b h n c
    q, k, v = hd(q), hd(k), hd(v)
    freqs = P["mid_attn.fn.fn.rotary_emb.freqs"]
    q = rope(q, freqs)
    k = rope(k, freqs)
    sim = torch.einsum("bhid,bhjd->bhij", q, k) * (DIM_HEAD ** -0.5)
    attn = sim.softmax(dim=-1)
    out = torch.einsum("bhij,bhjd->bhid", attn, v)
    out = out.permute(0, 1, 3, 2).reshape(b, HEADS * DIM_HEAD, n)
    out = F.conv1d(out, P["mid_attn.fn.fn.to_out.weight"], P["mid_attn.fn.fn.to_out.bias"])
    return out + x


# ----------------------------------------------------------------------------- denoiser (a6, a11)
def unet_forward(P, cfg, x, time, init_cond, attn_cond):
    """model/unet1d.py:1086-1166, simple=True, conditional=True branches, batched semantics.
    x, init_cond: (b, rt, mz); time: (b,) int64; attn_cond: (b, rt).  Returns (b, rt, mz)."""
    dim = cfg["dim"]
    n_levels = len(cfg["dim_mults"])
    b, rt, mz = x.shape
    R = b * rt
    x = x.reshape(R, 1, mz)
    t = time_mlp(P, time, dim)  # (b, 4*dim)

    # ConditionalScaleShift on the MS2-mixture channel (unet1d.py:666-678, 1107-1115)
    ss = F.linear(F.silu(t), P["init_cond_proj.to_scale_shift.1.weight"], P["init_cond_proj.to_scale_shift.1.bias"])
    ss = ss.repeat_interleave(rt, dim=0)  # (R, 2)
    ic = init_cond.reshape(R, 1, mz) * (ss[:, 0:1, None] + 1) + ss[:, 1:2, None]
    x = torch.cat((ic, x), dim=1)
    x = F.conv1d(x, P["init_conv.weight"], P["init_conv.bias"], padding=3)
    r = x

    # MS1 chromatogram -> (b, 8, rt)  (unet1d.py:1120-1130; mz_net is Identity)
    ac = attn_cond.reshape(b, 1, rt)
    ac = F.conv1d(ac, P["attn_cond_proj.1.0.weight"], P["attn_cond_proj.1.0.bias"], padding=3)
    ac = F.gelu(ac)
    ac = F.conv1d(ac, P["attn_cond_proj.1.2.weight"], P["attn_cond_proj.1.2.bias"])

    h = []
    for i in range(n_levels):
        pre = f"downs.{i}"
        x = resnet_block(P, pre + ".0", x, t, rt)
        h.append(x)
        x = resnet_block(P, pre + ".1", x, t, rt)
        x = linear_attention(P, pre + ".2", x)
        h.append(x)
        if i < n_levels - 1:
            x = F.conv1d(x, P[pre + ".3.weight"], P[pre + ".3.bias"], stride=2, padding=1)
        else:
            x = F.conv1d(x, P[pre + ".3.weight"], P[pre + ".3.bias"], padding=1)

    d, mzd = x.shape[1], x.shape[2]
    x = x.reshape(b, rt, d, mzd).permute(0, 2, 3, 1).reshape(b, d * mzd, rt)  # "(b rt) d mz -> b (d mz) rt"
    x = resnet_block(P, "mid_block1", x, t, 1)
    x = mid_attention(P, x, ac)
    x = resnet_block(P, "mid_block2", x, t, 1)
    x = x.reshape(b, d, mzd, rt).permute(0, 3, 1, 2).reshape(R, d, mzd)  # "b (d mz) rt -> (b rt) d mz"

    for j in range(n_levels):
        pre = f"ups.{j}"
        x = torch.cat((x, h.pop()), dim=1)
        x = resnet_block(P, pre + ".0", x, t, rt)
        x = torch.cat((x, h.pop()), dim=1)
        x = resnet_block(P, pre + ".1", x, t, rt)
        x = linear_attention(P, pre + ".2", x)
        if j < n_levels - 1:
            x = F.interpolate(x, scale_factor=2, mode="nearest")
            x = F.conv1d(x, P[pre + ".3.1.weight"], P[pre + ".3.1.bias"], padding=1)
        else:
            x = F.conv1d(x, P[pre + ".3.weight"], P[pre + ".3.bias"], padding=1)

    x = torch.cat((x, r), dim=1)
    x = resnet_block(P, "final_res_block", x, t, rt)
    x = F.conv1d(x, P["final_conv.weight"], P["final_conv.bias"])
    return x.reshape(b, rt, mz)


# ----------------------------------------------------------------------------- parameter inventory
def param_shapes(cfg):
    """Names and shapes of the reference's UNet1d.state_dict() for simple=True, conditional=True
    (model/unet1d.py:940-1084; key pattern in SURVEY.md §8b).  Returns an ordered dict name -> shape."""
    dim = cfg["dim"]
    mults = list(cfg["dim_mults"])
    dsd = cfg["downsample_dim"]
    td = dim * 4
    dims = [dim] + [dim * m for m in mults]
    in_out = list(zip(dims[:-1], dims[1:]))
    S = {}

    def conv(name, co, ci, k, bias=True):
        S[name + ".weight"] = (co, ci, k)
        if bias:
            S[name + ".bias"] = (co,)

    def lin(name, o, i):
        S[name + ".weight"] = (o, i)
        S[name + ".bias"] = (o,)

    def resblock(name, ci, co):
        lin(name + ".mlp.1", 2 * co, td)
        conv(name + ".block1.proj", co, ci, 3)
        S[name + ".block1.norm.g"] = (1, co, 1)
        conv(name + ".block2.proj", co, co, 3)
        S[name + ".block2.norm.g"] = (1, co, 1)
        if ci != co:
            conv(name + ".res_conv", co, ci, 1)

    def linattn(name, c):
        S[name + ".fn.fn.to_qkv.weight"] = (3 * HEADS * DIM_HEAD, c, 1)
        conv(name + ".fn.fn.to_out.0", c, HEADS * DIM_HEAD, 1)
        S[name + ".fn.fn.to_out.1.g"] = (1, c, 1)
        S[name + ".fn.norm.g"] = (1, c, 1)

    cin = cfg["channels"] + cfg["init_cond_channels"]
    conv("init_conv", dim, cin, 7)
    lin("time_mlp.1", td, dim)
    lin("time_mlp.3", td, td)
    lin("init_cond_proj.to_scale_shift.1", 2 * cfg["init_cond_channels"], td)
    acd = dim * 2
    conv("attn_cond_proj.1.0", acd, cfg["attn_cond_channels"], 7)
    conv("attn_cond_proj.1.2", acd, acd, 1)
    n = len(in_out)
    for i, (di, do) in enumerate(in_out):
        resblock(f"downs.{i}.0", di, di)
        resblock(f"downs.{i}.1", di, di)
        linattn(f"downs.{i}.2", di)
        conv(f"downs.{i}.3", do, di, 4 if i < n - 1 else 3)
    for j, (di, do) in enumerate(reversed(in_out)):
        resblock(f"ups.{j}.0", do + di, do)
        resblock(f"ups.{j}.1", do + di, do)
        linattn(f"ups.{j}.2", do)
        conv(f"ups.{j}.3.1" if j < n - 1 else f"ups.{j}.3", di, do, 3)
    dn = dsd // (2 ** (len(mults) - 1))
    cm = dims[-1] * dn
    resblock("mid_block1", cm, cm)
    S["mid_attn.fn.fn.rotary_emb.freqs"] = (DIM_HEAD // 4,)
    S["mid_attn.fn.fn.to_qv.weight"] = (2 * HEADS * DIM_HEAD, cm, 1)
    S["mid_attn.fn.fn.to_k.weight"] = (HEADS * DIM_HEAD, acd, 1)
    conv("mid_attn.fn.fn.to_out", cm, HEADS * DIM_HEAD, 1)
    S["mid_attn.fn.norm.g"] = (1, cm, 1)
    resblock("mid_block2", cm, cm)
    resblock("final_res_block", dim * 2, dim)
    conv("final_conv", cfg["channels"], dim, 1)
    return S


def rotary_freqs():
    d = DIM_HEAD // 2
    return 1.0 / (10000 ** (torch.arange(0, d, 2)[: d // 2].float() / d))


def det_tensor(name, shape, scale=1.0, seed=0):
    """Deterministic pseudo-random tensor from a name (shared by gen_golden.py, tests and bench so that no
    weights have to be committed): torch CPU generator seeded with crc32(name) ^ seed."""
    import zlib

    g = torch.Generator(device="cpu")
    g.manual_seed((zlib.crc32(name.encode()) ^ (seed * 0x9E3779B1)) & 0x7FFFFFFF)
    return torch.randn(shape, generator=g, dtype=torch.float32) * scale


def det_params(cfg, seed=0):
    """Deterministic parameters with the reference's shapes.  Magnitudes follow PyTorch's default init
    scale (uniform(-1/sqrt(fan_in), 1/sqrt(fan_in)) has std 1/sqrt(3*fan_in)); g = 1 + small noise so
    that the norm gains are exercised."""
    P = {}
    for name, shape in param_shapes(cfg).items():
        if name.endswith("rotary_emb.freqs"):
            P[name] = rotary_freqs()
        elif name.endswith(".g"):
            P[name] = 1.0 + det_tensor(name, shape, 0.1, seed)
        elif name.endswith(".bias"):
            P[name] = det_tensor(name, shape, 0.05, seed)
        else:
            fan_in = 1
            for s in shape[1:]:
                fan_in *= s
            P[name] = det_tensor(name, shape, 1.0 / math.sqrt(fan_in), seed)
    return P


# ----------------------------------------------------------------------------- training step (a4, a12)
def train_loss(P, cfg, alpha_bars, x0, ms2_cond, ms1_cond, t, noise):
    """model/model.py:343-404 with pred_type='eps', auto_normalize=True, ms1_loss_weight=0; `t` and `noise`
    injected (noise is the N(0,1) tensor itself, i.e. what the reference draws at model.py:346)."""
    x0n = normalize(x0)
    c2 = normalize(ms2_cond)
    c1 = normalize(ms1_cond)
    x_t = q_sample(alpha_bars, x0n, t, noise)
    eps = unet_forward(P, cfg, x_t, t, c2, c1)
    return F.mse_loss(eps, noise), eps


def clip_grad_norm(grads, max_norm=10.0):
    """torch.nn.utils.clip_grad_norm_ (model/model_interface.py:1121): global L2, coef = min(1, max/(norm+1e-6))."""
    total = torch.sqrt(sum((g.double() ** 2).sum() for g in grads)).float()
    coef = torch.clamp(max_norm / (total + 1e-6), max=1.0)
    return [g * coef for g in grads], total


def adamw_step(p, g, m, v, step, lr, b1=0.9, b2=0.999, eps=1e-8, wd=0.01):
    """torch.optim.AdamW defaults (model/model_interface.py:1011), single-tensor formulation."""
    p = p * (1 - lr * wd)
    m = m + (1 - b1) * (g - m)  # lerp
    v = v * b2 + (1 - b2) * g * g
    bc1 = 1 - b1 ** step
    bc2 = 1 - b2 ** step
    denom = (v.sqrt() / math.sqrt(bc2)) + eps
    p = p - (lr / bc1) * m / denom
    return p, m, v


def lr_lambda(epoch, warmup, total):
    """model/model_interface.py:149-155 (num_cycles = 0.5)."""
    if epoch < warmup:
        return float(epoch + 1) / float(max(1, warmup))
    prog = float(epoch - warmup) / float(max(1, total - warmup))
    return max(1e-10, 0.5 * (1.0 + math.cos(math.pi * 0.5 * 2.0 * prog)))


# ----------------------------------------------------------------------------- secondary modes (SURVEY §8f-3)
def sic_loss(x0_like, ms1_cond_n):
    """MS1 summary-ion-chromatogram loss, model/model.py:364-371 / 379-386 — DEFINED HERE, not restated: the reference
    loops `func in (torch.sum, torch.mean, torch.max)` with `dim=-1`; `torch.max(x, dim=-1)` returns a (values, indices)
    tuple, so the reference raises TypeError whenever ms1_loss_weight > 0, and its `func(ms1_cond, dim=-1)` would
    reduce the (b, RT) chromatogram to (b,).  The evident intent — compare the RT profile of the predicted map with
    the MS1 chromatogram — is what is implemented: for each reduction f in (sum, mean, max-values) over the mz axis,
    sic_f = f(x0_like) of shape (b, RT); both profiles are divided by their global maximum (as the reference does)
    and compared with an MSE over all (b, RT) entries; the three terms add up."""
    total = x0_like.new_zeros(())
    tgt = ms1_cond_n / torch.max(ms1_cond_n)
    for f in (lambda v: v.sum(-1), lambda v: v.mean(-1), lambda v: v.max(-1).values):
        sic = f(x0_like)
        total = total + F.mse_loss(sic / torch.max(sic), tgt)
    return total


def train_loss_modes(P, cfg, alpha_bars, x0, ms2_cond, ms1_cond, t, noise, pred_type="eps", ms1_loss_weight=0.0,
                     pos_output_only=False):
    """model/model.py:343-404 for every (pred_type, ms1_loss_weight, pos_output_only) combination; returns the (b,)
    loss vector of the batched semantics (batch-mean primary loss times loss_weight[t_i]) and the network output."""
    x0n = normalize(x0)
    c2 = normalize(ms2_cond)
    c1 = normalize(ms1_cond)
    x_t = q_sample(alpha_bars, x0n, t, noise)
    out = unet_forward(P, cfg, x_t, t, c2, c1)
    if pos_output_only:
        out = F.softplus(out)                      # model/unet1d.py:1084, 1166
    if pred_type == "eps":
        primary = F.mse_loss(out, noise)
        x0_like = x_t - out                        # model/model.py:367 (the reference's choice, not (x_t - s eps)/a)
    elif pred_type == "x0":
        primary = F.mse_loss(out, x0n)
        x0_like = out
    else:
        raise ValueError(f"Unknown pred_type: {pred_type}")
    loss = primary
    if ms1_loss_weight > 0.0:
        loss = (1 - ms1_loss_weight) * primary + ms1_loss_weight * sic_loss(x0_like, c1)
    return loss * loss_weight_table(alpha_bars, pred_type)[t], out


def ddim_update_x0(alpha_bars, x_t, x0_pred, t):
    """model/model.py:275-289, pred_type == 'x0'."""
    ab = alpha_bars[t]
    eps = (x_t - torch.sqrt(ab) * x0_pred) / torch.sqrt(1.0 - ab)
    if t > 0:
        abp = alpha_bars[t - 1]
        return torch.sqrt(abp) * x0_pred + torch.sqrt(1.0 - abp) * eps, eps
    return x0_pred, eps


# ----------------------------------------------------------------------------- sampling (a5)
def ddim_sample(P, cfg, alpha_bars, x_T, ms2_cond, ms1_cond, num_steps):
    """model/model.py:293-324."""
    T = alpha_bars.shape[0]
    c2 = normalize(ms2_cond)
    c1 = normalize(ms1_cond)
    x = x_T
    b = x.shape[0]
    for t in ddim_timesteps(T, num_steps):
        ti = int(t.item())
        eps = unet_forward(P, cfg, x, torch.full((b,), ti, dtype=torch.long), c2, c1)
        x = ddim_update(alpha_bars, x, eps, ti)
    x = unnormalize(x)
    pred_noise = unnormalize(c2) - x
    return x, pred_noise


# ----------------------------------------------------------------------------- data (a13, a14)
def pair_draw(rng, n, used):
    """utils/data_loader.py:111-125: rejection loop over python `random`."""
    while True:
        i1 = rng.randint(0, n - 1)
        i2 = rng.randint(0, n - 1)
        if i1 == i2:
            continue
        pair = tuple(sorted((i1, i2)))
        if pair in used:
            continue
        used.add(pair)
        return i1, i2


def minmax_pair(ms2_1, ms1_1, ms2_2, ms1_2):
    """utils/data_loader.py:70-88 on numpy arrays; returns 4 float32 numpy arrays."""
    import numpy as np

    ms2_min = np.min([ms2_1.min(), ms2_2.min()])
    ms2_max = np.max([ms2_1.max(), ms2_2.max()])
    ms1_min = np.min([ms1_1.min()])
    ms1_max = np.max([ms1_1.max()])
    a = (ms2_1 - ms2_min) / (ms2_max - ms2_min)
    b = (ms1_1 - ms1_min) / (ms1_max - ms1_min)
    c = (ms2_2 - ms2_min) / (ms2_max - ms2_min)
    d = (ms1_2 - ms1_min) / (ms1_max - ms1_min)
    return tuple(z.astype(np.float32) for z in (a, b, c, d))


def mix(ms2_1, ms2_2, w=(0.5, 0.5)):
    """model/model_interface.py:1073-1075."""
    return ms2_1 * w[0] + ms2_2 * w[1]
