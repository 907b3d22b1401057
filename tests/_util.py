import math
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "diffusion-deconvolution-dia-msms-data_b200"), os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

TINY = dict(dim=4, channels=1, dim_mults=[1, 2, 2, 3, 3, 4, 4], conditional=True, init_cond_channels=1,
            attn_cond_channels=1, tfer_dim_mult=620, downsample_dim=320, simple=True)


def make_net(cfg=TINY, seed=0, device="cuda"):
    """B200 UNet1d with the oracle's deterministic parameters loaded; returns (net, P_cpu)."""
    import dquartic_oracle as O
    from dquartic.model.unet1d import UNet1d

    net = UNet1d(dim=cfg["dim"], channels=1, dim_mults=tuple(cfg["dim_mults"]), conditional=True,
                 init_cond_channels=1, attn_cond_channels=1, downsample_dim=cfg["downsample_dim"], simple=True)
    P = O.det_params(cfg, seed)
    net.load_state_dict(P)
    return net.to(device), P


def rel_err(a, b):
    a = a.detach().float().cpu()
    b = b.detach().float().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-12))


def golden(name):
    return np.load(os.path.join(ROOT, "tests", "golden", name))


# ---------------------------------------------------------------------------------------------- per-element checks
U = 2.0 ** -24          # fp32 unit roundoff
NAN = float("nan")


def _nan(*shape, dtype=torch.float32):
    return torch.full(shape, NAN, dtype=dtype, device="cuda")


def _nan_empty(net):
    """Make net._empty return NaN-filled tensors (an element a kernel should write but does not stays NaN)."""
    def empty(*shape, dtype=torch.float32):
        return torch.full(shape, NAN, dtype=dtype, device=net._flat.device)
    net._empty = empty


def _restore_empty(net):
    net.__dict__.pop("_empty", None)


def _check(tag, got, ref, bound, rt=None, row0=0):
    """Every element within its bound (a NaN fails).  Prints the worst error / bound.  For an (R, C, L) activation
    with `rt` rows per sample (`row0`: first row of this slice) the first failing element is named as sample, row,
    channel and position."""
    err = (got.double() - ref).abs()
    ok = err <= bound
    if not bool(ok.all()):
        bad = (~ok).nonzero()
        i = tuple(bad[0].tolist())
        where = ""
        if rt is not None and got.dim() == 3:
            r = row0 + i[0]
            where = f" = sample {r // rt}, row {r % rt}, channel {i[1]}, position {i[2]} of {got.shape[2]}"
        raise AssertionError(f"{tag}: {bad.shape[0]} of {ok.numel()} elements out of bound; first {i}{where}: "
                             f"got {float(got[i])}, ref {float(ref[i])}, bound {float(bound[i])}")
    frac = float((err / bound.clamp_min(1e-300)).max())
    print(f"BOUND {tag}: max err / bound = {frac:.3g}")
    return frac


def _exp_ulp(x):
    """CUDA Programming Guide, intrinsic functions: __expf(x) has a maximum error of 2 + floor(|1.173 x|) ulp."""
    return 2 + torch.floor((1.173 * x).abs())


def _act_ref(z, act):
    if act == 1:
        return z * torch.sigmoid(z), torch.sigmoid(z) * (1 + z * (1 - torch.sigmoid(z)))
    if act == 2:
        cdf = 0.5 * (1 + torch.erf(z / math.sqrt(2)))
        return z * cdf, cdf + z * torch.exp(-0.5 * z * z) / math.sqrt(2 * math.pi)
    if act == 3:
        sp = torch.where(z > 20, z, torch.log1p(torch.exp(z)))
        return sp, torch.where(z > 20, torch.ones_like(z), torch.sigmoid(z))
    return z, torch.ones_like(z)


def _act_bounds(z, act):
    """Per-element absolute error bounds of the kernel's fp32 act_fwd / act_bwd (csrc/common.cuh).
    SiLU and the GELU derivative use __expf, whose error the CUDA Programming Guide bounds by 2 + floor(|1.173 x|) ulp;
    expf, erff and log1pf are within 2 ulp."""
    za = z.abs()
    if act == 1:
        e1 = U * (_exp_ulp(z) + 4)
        s = torch.sigmoid(z)
        return 2 * e1 * (z * s).abs(), 2 * (e1 + 4 * U) * s * (1 + za * (1 + s))
    if act == 2:
        erf = torch.erf(z / math.sqrt(2)).abs()
        pdf = torch.exp(-0.5 * z * z) / math.sqrt(2 * math.pi)
        fwd = 6 * U * 0.5 * za * (1 + erf)
        e2 = U * (_exp_ulp(0.5 * z * z) + z * z + 4)
        return fwd, 2 * (4 * U * (1 + erf) + za * pdf * e2)
    if act == 3:
        E = torch.exp(torch.clamp(z, max=20))
        sp, dsp = _act_ref(z, 3)
        small = z <= 20
        fwd = torch.where(small, U * (4 * E / (1 + E) + 3 * sp.abs()), torch.zeros_like(z))
        return fwd, torch.where(small, 6 * U * dsp.abs(), torch.zeros_like(z))
    return torch.zeros_like(z), torch.zeros_like(z)


def _misaligned(t):
    """A contiguous copy of `t` whose base address is 4 bytes past a 16-byte boundary (kernels must leave their vector paths)."""
    flat = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    v = flat[1:].view(t.shape)
    v.copy_(t)
    assert v.is_contiguous() and v.data_ptr() % 16 == 4
    return v
