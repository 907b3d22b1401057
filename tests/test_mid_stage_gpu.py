"""GPU: the tcgen05 GEMM and the mid-stage kernels element by element, at the shapes training runs
(micro-batch 64, RT 34, 10000 mid channels), against float64 references computed on the GPU.

Every comparison is per element against a bound derived from the kernel's arithmetic (u = 2^-24, the fp32 unit
roundoff); outputs that are not accumulated are pre-filled with NaN, so an element the kernel never wrote fails.
`pytest -s` prints the largest observed error of each check as a fraction of its bound."""
import math

import pytest
import torch
import torch.nn.functional as F

from _util import TINY, make_net

pytestmark = pytest.mark.gpu

U = 2.0 ** -24          # fp32 unit roundoff
UB = 2.0 ** -8          # bf16 unit roundoff (round to nearest)
GEMM_REL = 1e-5         # |C - R| <= 1e-5 * (|A| . |B|^T + |bias| + |C_old|)
HD, HEADS = 128, 4
NAN = float("nan")
BIG = dict(TINY, downsample_dim=40000)   # mid channels 16 * 625 = 10000


# ---------------------------------------------------------------------------------------------- helpers
def _nan(*shape, dtype=torch.float32):
    return torch.full(shape, NAN, dtype=dtype, device="cuda")


def _check(tag, got, ref, bound):
    """Every element within its bound (a NaN fails).  Prints the worst error / bound."""
    err = (got.double() - ref).abs()
    ok = err <= bound
    if not bool(ok.all()):
        bad = (~ok).nonzero()
        i = tuple(bad[0].tolist())
        raise AssertionError(f"{tag}: {bad.shape[0]} of {ok.numel()} elements out of bound; first {i}: "
                             f"got {float(got[i])}, ref {float(ref[i])}, bound {float(bound[i])}")
    frac = float((err / bound.clamp_min(1e-300)).max())
    print(f"BOUND {tag}: max err / bound = {frac:.3g}")
    return frac


def _shift(A, o):
    """A_tap[m] = A[m + o], zero outside (TMA's out-of-range fill)."""
    if o == 0:
        return A
    R = torch.zeros_like(A)
    if o > 0:
        R[:-o] = A[o:]
    else:
        R[-o:] = A[:o]
    return R


def _pick_bn(m_tiles, N, nz, sms):
    """Host-side tile width choice of dq_gemm_bf16_tn (csrc/gemm_tcgen05.cu: pick_bn), restated to report it."""
    if N <= 128:
        return 128
    if N <= 256:
        return 256
    best, best_cost = 256, 1e30
    for bn in range(256, 127, -16):
        tiles = m_tiles * ((N + bn - 1) // bn) * nz
        cost = ((tiles + sms - 1) // sms) * (bn + 24)
        if cost < best_cost * 0.995:
            best_cost, best = cost, bn
    return best


def _report_bn(tag, M, N, nz=1):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    print(f"PICK_BN {tag}: M={M} N={N} nz={nz} -> bn {_pick_bn((M + 127) // 128, N, nz, sms)}")


def _nan_empty(net):
    """Make net._empty return NaN-filled tensors (an element a kernel should write but does not stays NaN)."""
    def empty(*shape, dtype=torch.float32):
        return torch.full(shape, NAN, dtype=dtype, device=net._flat.device)
    net._empty = empty


def _restore_empty(net):
    net.__dict__.pop("_empty", None)


@pytest.fixture(scope="module")
def tiny():
    from dquartic import _native as N
    net, _ = make_net()
    net._refresh_bf16()
    net._ensure_grads()
    return net, N


@pytest.fixture(scope="module")
def big():
    """10000-channel mid stage; parameters drawn on the device from a seeded generator (default init), norm gains
    perturbed away from 1 so that a dropped gain shows."""
    from dquartic import _native as N
    from dquartic.model.unet1d import UNet1d
    torch.cuda.manual_seed(1234)
    net = UNet1d(dim=BIG["dim"], channels=1, dim_mults=tuple(BIG["dim_mults"]), conditional=True, init_cond_channels=1,
                 attn_cond_channels=1, downsample_dim=BIG["downsample_dim"], simple=True, device="cuda")
    assert net.mid_channels == 10000
    g = torch.Generator(device="cuda").manual_seed(99)
    with torch.no_grad():
        for name in net.specs:
            if name.endswith(".g"):
                w = net._w(name)
                w.copy_(1 + 0.3 * torch.randn(w.shape, generator=g, device="cuda"))
    net.mark_params_modified()
    net._refresh_bf16()
    net._ensure_grads()
    yield net, N
    net._wgrad_defer = None


def _net_for(N_ch, tiny, big):
    return big if N_ch == 10000 else tiny


# ---------------------------------------------------------------------------------------------- 1. GEMM
def _conv_ref(Ap, W3, offs, bias=None):
    """sum_t shift(A, offs[t]) . W3[t]^T (+ bias) and the matching |.| product, in float64 on the GPU."""
    A = Ap.double()
    R = torch.zeros(A.shape[0], W3.shape[1], dtype=torch.float64, device="cuda")
    M = torch.zeros_like(R)
    for t, o in enumerate(offs):
        Wt = W3[t].double()
        As = _shift(A, o)
        R += As @ Wt.T
        M += As.abs() @ Wt.abs().T
        del Wt, As
    if bias is not None:
        R += bias.double()
        M += bias.double().abs()
    return R, M


@pytest.mark.parametrize("b,rt,Nch", [(64, 34, 10000), (7, 136, 10000), (1, 34, 10000), (3, 5, 80)])
def test_gemm_mid_conv_fwd_dgrad(tiny, big, b, rt, Nch):
    """The RT convolution forward (taps -1, 0, 1 with bias) and data gradient (taps 1, 0, -1) exactly as
    _mid_conv_fwd / _mid_conv_dgrad issue them; every padded row (halo rows included) is checked."""
    net, N = _net_for(Nch, tiny, big)
    assert net.mid_channels == Nch
    wname, bname = "mid_block1.block1.proj.weight", "mid_block1.block1.proj.bias"
    Mp = b * (rt + 2)
    g = torch.Generator(device="cuda").manual_seed(b * 1000 + rt)
    X = torch.randn(b * rt, Nch, generator=g, device="cuda")
    Ap = _nan(Mp, Nch, dtype=torch.bfloat16)
    N.call("dq_mid_pack", X, Ap, b, rt, Nch, 1)
    W3, WT3, bias = net._bf16[wname], net._bf16[wname + ".T"], net._w(bname)
    R, Mag = _conv_ref(Ap, W3, (-1, 0, 1), bias)
    bns = (0, 128, 208, 256) if (b, rt) == (64, 34) else (0,)
    _report_bn(f"conv b={b} rt={rt}", Mp, Nch)
    _nan_empty(net)
    try:
        for bn in bns:
            net.gemm_bn = bn
            Uo = net._mid_conv_fwd(Ap, wname, bname, b, rt)
            torch.cuda.synchronize()
            assert N.gemm_last_error() == 0
            _check(f"conv fwd b={b} rt={rt} N={Nch} bn={bn}", Uo, R, GEMM_REL * Mag)
        del R, Mag
        dU = torch.randn(b * rt, Nch, generator=g, device="cuda")
        dUp = _nan(Mp, Nch, dtype=torch.bfloat16)
        N.call("dq_mid_pack", dU, dUp, b, rt, Nch, 1)
        R, Mag = _conv_ref(dUp, WT3, (1, 0, -1))
        for bn in bns:
            net.gemm_bn = bn
            dX = net._mid_conv_dgrad(dUp, wname, b, rt)
            torch.cuda.synchronize()
            assert N.gemm_last_error() == 0
            _check(f"conv dgrad b={b} rt={rt} N={Nch} bn={bn}", dX, R, GEMM_REL * Mag)
    finally:
        net.gemm_bn = 0
        _restore_empty(net)


def _wgrad_ref(pairs, C_old):
    """dW[t] = C_old[t] + sum over micro-batches of dU^T . shift(A, t - 1) (per micro-batch shift), and |.|."""
    R = C_old.double().clone()
    Mag = C_old.double().abs()
    for dUp, Ap in pairs:
        dT = dUp.double().T.contiguous()
        A = Ap.double()
        for t in range(3):
            As = _shift(A, t - 1)
            R[t] += dT @ As
            Mag[t] += dT.abs() @ As.abs()
            del As
    return R, Mag


def test_gemm_mid_conv_wgrad_unplanned_planned_and_union(big):
    """The weight gradient as _mid_conv_wgrad issues it (nz = 3, z_b_tap_step = 1, z_c_stride = N*N, accumulate):
    once unplanned (K = Mp = 2304), once through a 4-micro-batch _wgrad_defer plan (K = 4 Mp = 9216), and once as a
    single pass over the union batch (b = 256).  All three within the bound of the float64 reference."""
    net, N = big
    Nch = net.mid_channels
    wname = "mid_block2.block1.proj.weight"
    b, rt = 64, 34
    Mp = b * (rt + 2)
    g = torch.Generator(device="cuda").manual_seed(7)
    pairs = []
    for _ in range(4):
        dUp = _nan(Mp, Nch, dtype=torch.bfloat16)
        Ap = _nan(Mp, Nch, dtype=torch.bfloat16)
        N.call("dq_mid_pack", torch.randn(b * rt, Nch, generator=g, device="cuda"), dUp, b, rt, Nch, 1)
        N.call("dq_mid_pack", torch.randn(b * rt, Nch, generator=g, device="cuda"), Ap, b, rt, Nch, 1)
        pairs.append((dUp, Ap))
    C_old = torch.randn(3, Nch, Nch, generator=g, device="cuda")
    dW = net._gw(wname).view(3, Nch, Nch)
    _report_bn("wgrad K=2304", Nch, Nch, 3)
    _report_bn("wgrad K=9216", Nch, Nch, 3)
    _nan_empty(net)
    try:
        net._wgrad_defer = None
        dW.copy_(C_old)
        net._mid_conv_wgrad(pairs[0][0], pairs[0][1], wname, b, rt)
        torch.cuda.synchronize()
        assert N.gemm_last_error() == 0
        R, Mag = _wgrad_ref(pairs[:1], C_old)
        _check("wgrad unplanned K=2304", dW, R, GEMM_REL * Mag)
        del R, Mag
        dW.copy_(C_old)
        net._wgrad_stash = {}
        for i, (dUp, Ap) in enumerate(pairs):
            net._wgrad_defer = (i * Mp, 4 * Mp, i == 3)
            net._mid_conv_wgrad(dUp, Ap, wname, b, rt)
        net._wgrad_defer = None
        net._wgrad_stash = {}
        torch.cuda.synchronize()
        assert N.gemm_last_error() == 0
        planned = dW.clone()
        R, Mag = _wgrad_ref(pairs, C_old)
        _check("wgrad planned 4x64 K=9216", planned, R, GEMM_REL * Mag)
        dW.copy_(C_old)
        dU_all = torch.cat([p[0] for p in pairs])
        A_all = torch.cat([p[1] for p in pairs])
        net._mid_conv_wgrad(dU_all, A_all, wname, 4 * b, rt)
        torch.cuda.synchronize()
        assert N.gemm_last_error() == 0
        _check("wgrad union b=256 K=9216", dW, R, GEMM_REL * Mag)
        _check("wgrad planned vs union", planned, dW.double(), GEMM_REL * Mag)
    finally:
        net._wgrad_defer = None
        net._wgrad_stash = {}
        net._gflat.zero_()
        _restore_empty(net)


@pytest.mark.parametrize("kind", ["qv", "out", "dO", "dxn", "dWout", "dWqv"])
def test_gemm_mid_attention_shapes(big, kind):
    """The six GEMMs of _mid_attn_fwd / _mid_attn_bwd at b = 64, rt = 34 (M = 2176) with their operands:
    N = 256 and K = Nm; bias + accumulate into a prefilled C; the wout.T and wqv.T operands; the two accumulated
    weight gradients with K = M."""
    net, N = big
    Nm = net.mid_channels
    M = 64 * 34
    g = torch.Generator(device="cuda").manual_seed(11)

    def rb(*shape):
        return torch.randn(shape, generator=g, device="cuda").bfloat16()

    bias, acc, C_old = None, 0, None
    if kind == "qv":        # qv = xn . Wqv^T
        A, B, Mr, Nn, K = rb(M, Nm), net._bf16["wqv"], M, 2 * HD, Nm
    elif kind == "out":     # out = X + O . Wout^T + b
        A, B, Mr, Nn, K = rb(M, HD), net._bf16["wout"], M, Nm, HD
        bias, acc = net._w("mid_attn.fn.fn.to_out.bias"), 1
        C_old = torch.randn(M, Nm, generator=g, device="cuda")
    elif kind == "dO":      # dO = dOut . Wout
        A, B, Mr, Nn, K = rb(M, Nm), net._bf16["wout.T"], M, HD, Nm
    elif kind == "dxn":     # dxn = dqv . Wqv
        A, B, Mr, Nn, K = rb(M, 2 * HD), net._bf16["wqv.T"], M, Nm, 2 * HD
    elif kind == "dWout":   # dWout += dOut^T . O
        A, B, Mr, Nn, K, acc = rb(Nm, M), rb(HD, M), Nm, HD, M, 1
        C_old = torch.randn(Nm, HD, generator=g, device="cuda")
    else:                   # dWqv += dqv^T . xn
        A, B, Mr, Nn, K, acc = rb(2 * HD, M), rb(Nm, M), 2 * HD, Nm, M, 1
        C_old = torch.randn(2 * HD, Nm, generator=g, device="cuda")
    Ad, Bd = A.double(), B.double()
    R = Ad @ Bd.T
    Mag = Ad.abs() @ Bd.abs().T
    if bias is not None:
        R += bias.double()
        Mag += bias.double().abs()
    if C_old is not None:
        R += C_old.double()
        Mag += C_old.double().abs()
    C = C_old.clone() if acc else _nan(Mr, Nn)
    _report_bn(f"attn {kind}", Mr, Nn)
    net.gemm_bn = 0
    net._gemm(A, Mr, K, K, B, Nn, K, K, 0, 1, C, Nn, bias, acc, Mr, Nn, K, 1, (0,), (0,), (0,), (0,))
    torch.cuda.synchronize()
    assert N.gemm_last_error() == 0
    _check(f"attn gemm {kind}", C, R, GEMM_REL * Mag)


# ---------------------------------------------------------------------------------------------- 2. fp32 kernels
def _exp_ulp(x):
    """CUDA Programming Guide, intrinsic functions: __expf(x) has a maximum error of 2 + floor(|1.173 x|) ulp."""
    return 2 + torch.floor((1.173 * x).abs())


# (ss, act, upad, dhpad, opad, du mode): du mode "bf16" = padded/plain bf16 output, "f32" = fp32 output,
# "f32acc" = accumulate into fp32, "both" = fp32 + bf16.  dg, dbias and (with ss) dss are always accumulated.
ROWNORM_CASES = [
    (True, 1, 1, 1, 1, "bf16"),      # mid block1 backward
    (False, 1, 1, 0, 1, "bf16"),     # mid block2 backward
    (False, 0, 0, 0, 0, "f32acc"),   # mid attention PreNorm backward
    (True, 0, 0, 1, 0, "both"),
    (False, 1, 1, 1, 0, "f32acc"),
    (True, 1, 0, 0, 0, "f32"),
]


@pytest.mark.parametrize("b,rt,Nch", [(64, 34, 10000), (5, 7, 1030)])
@pytest.mark.parametrize("case", ROWNORM_CASES)
def test_rownorm_bwd_against_float64(tiny, b, rt, Nch, case):
    _, N = tiny
    ss_on, act, upad, dhpad, opad, mode = case
    M = b * rt
    Mp = b * (rt + 2)
    g = torch.Generator(device="cuda").manual_seed(Nch + 17 * act + 3 * upad + dhpad)
    dev = "cuda"

    def padded(valid, pad):   # halo rows NaN: a kernel that reads them fails
        if not pad:
            return valid.contiguous()
        out = _nan(Mp, Nch)
        out.view(b, rt + 2, Nch)[:, 1:rt + 1] = valid.view(b, rt, Nch)
        return out

    u = torch.randn(M, Nch, generator=g, device=dev) * 0.7
    u[rt + 3] = 0.0                                    # an all-zero row: the clamped-norm branch
    dh = torch.randn(M, Nch, generator=g, device=dev)
    gain = 1 + 0.3 * torch.randn(Nch, generator=g, device=dev)
    stride = 2 * Nch + 6
    SS = 0.5 * torch.randn(b, stride, generator=g, device=dev)
    dSS0 = torch.randn(b, stride, generator=g, device=dev)
    dSS = dSS0.clone()
    col = 2                                            # producers start at an even column of SS
    inv = (1.0 / u.double().norm(dim=1).clamp_min(1e-12)).float()
    dg0 = torch.randn(Nch, generator=g, device=dev)
    db0 = torch.randn(Nch, generator=g, device=dev)
    dg, dbias = dg0.clone(), db0.clone()
    dot = _nan(M)
    du_bf = _nan(Mp if opad else M, Nch, dtype=torch.bfloat16) if mode in ("bf16", "both") else None
    du0 = torch.randn(M, Nch, generator=g, device=dev)
    du_f = (du0.clone() if mode == "f32acc" else _nan(M, Nch)) if mode != "bf16" else None
    ss_ptr = SS.data_ptr() + 4 * col if ss_on else None
    dss_ptr = dSS.data_ptr() + 4 * col if ss_on else None
    N.call("dq_rownorm_bwd", padded(dh, dhpad), dhpad, padded(u, upad), upad, gain, ss_ptr, stride if ss_on else 0,
           act, inv, dot, du_bf, opad, du_f, 1 if mode == "f32acc" else 0, dg, dss_ptr, dbias, b, rt, Nch)
    torch.cuda.synchronize()

    # float64 reference with torch F.normalize semantics (x / max(||x||, 1e-12)), autograd for the gradients
    ud = u.double().requires_grad_(True)
    gd = gain.double().requires_grad_(True)
    sc = SS[:, col:col + Nch].double().requires_grad_(True)
    sh = SS[:, col + Nch:col + 2 * Nch].double().requires_grad_(True)
    sq = math.sqrt(Nch)
    n = F.normalize(ud, dim=1) * gd * sq
    z = (n.view(b, rt, Nch) * (sc[:, None] + 1) + sh[:, None]).view(M, Nch) if ss_on else n
    h = F.silu(z) if act == 1 else z
    (h * dh.double()).sum().backward()
    R_du, R_dg = ud.grad, gd.grad

    # magnitudes: the same chain on absolute values (a derivative of SiLU that crosses zero has an absolute error)
    with torch.no_grad():
        uh = u.double() * inv.double()[:, None]
        nd = uh * gain.double() * sq
        sc1 = (sc.detach() + 1).repeat_interleave(rt, 0) if ss_on else torch.ones_like(nd)
        zd = nd * sc1 + (sh.detach().repeat_interleave(rt, 0) if ss_on else 0)
        if act == 1:
            s = torch.sigmoid(zd)
            amag = s * (1 + zd.abs() * (1 + s))
            c_act = float(_exp_ulp(zd).max()) + 4
        else:
            amag = torch.ones_like(zd)
            c_act = 0.0
        dzm = dh.double().abs() * amag
        duhm = dzm * sc1.abs() * gain.double().abs() * sq
        dotm = (duhm * uh.abs()).sum(1, keepdim=True)
        clamped = inv.double()[:, None] >= 1e12
        dum = inv.double()[:, None] * torch.where(clamped, duhm, duhm + uh.abs() * dotm)
        c_el = 16 + c_act
        c_du = c_el + Nch / 256 + 13                    # + depth of the row dot product (strided, warp, block)
        b_du = c_du * U * dum
        R_dbias = db0.double() + R_du.sum(0)
        b_dbias = (c_du + rt + b + 2) * U * (dum.sum(0) + db0.double().abs())
        b_dg = (c_el + rt + b + 2) * U * ((dzm * sc1.abs() * uh.abs()).sum(0) * sq + dg0.double().abs())
    tag = f"rownorm_bwd b={b} rt={rt} N={Nch} ss={ss_on} act={act} upad={upad} dhpad={dhpad} opad={opad} {mode}"
    if du_f is not None:
        ref = R_du + (du0.double() if mode == "f32acc" else 0)
        bnd = b_du + (c_el * U * du0.double().abs() if mode == "f32acc" else 0)
        _check(tag + " du_f32", du_f, ref, bnd)
    if du_bf is not None:
        valid = du_bf.view(b, rt + 2, Nch)[:, 1:rt + 1].reshape(M, Nch) if opad else du_bf
        _check(tag + " du_bf16", valid, R_du, b_du + UB * (R_du.abs() + b_du))
        if opad:   # the caller owns the halo rows: the kernel must not write them
            halo = du_bf.view(b, rt + 2, Nch)[:, [0, rt + 1]]
            assert torch.isnan(halo.float()).all(), tag + " wrote a halo row"
    _check(tag + " dg", dg, dg0.double() + R_dg, b_dg)
    _check(tag + " dbias", dbias, R_dbias, b_dbias)
    if ss_on:
        with torch.no_grad():
            dzs = dzm.view(b, rt, Nch)
            b_dsc = (c_el + rt + 2) * U * ((dzs * nd.abs().view(b, rt, Nch)).sum(1) + dSS0[:, col:col + Nch].double().abs())
            b_dsh = (c_el + rt + 2) * U * (dzs.sum(1) + dSS0[:, col + Nch:col + 2 * Nch].double().abs())
        _check(tag + " dscale", dSS[:, col:col + Nch], dSS0[:, col:col + Nch].double() + sc.grad, b_dsc)
        _check(tag + " dshift", dSS[:, col + Nch:col + 2 * Nch], dSS0[:, col + Nch:col + 2 * Nch].double() + sh.grad,
               b_dsh)
        # columns of SS outside this producer's range are never touched
        assert torch.equal(dSS[:, :col], dSS0[:, :col]) and torch.equal(dSS[:, col + 2 * Nch:], dSS0[:, col + 2 * Nch:])
    else:
        assert torch.equal(dSS, dSS0)


def _rope64(t, freqs):
    """float64 restatement of oracle.rope on (b, h, n, 32): interleaved pairs of the first 16 features rotated by
    n * freqs[p] (the angle is formed from the fp32 freqs the kernel reads)."""
    n = t.shape[-2]
    ang = torch.arange(n, dtype=torch.float64, device=t.device)[:, None] * freqs.double()[None, :]
    cs, sn = ang.cos(), ang.sin()
    x1, x2 = t[..., 0:16:2], t[..., 1:16:2]
    r1 = x1 * cs - x2 * sn
    r2 = x2 * cs + x1 * sn
    rot = torch.stack((r1, r2), dim=-1).flatten(-2)
    return torch.cat((rot, t[..., 16:]), dim=-1)


def _rope_mag(t):
    """|rotated value| <= |x1| + |x2| for the rotated pairs."""
    a = t.abs()
    pair = a[..., 0:16:2] + a[..., 1:16:2]
    return torch.cat((torch.stack((pair, pair), dim=-1).flatten(-2), a[..., 16:]), dim=-1)


@pytest.mark.parametrize("rt", [1, 5, 31, 33, 34, 64, 136, 140])
def test_attn_core_fwd_bwd_against_float64(tiny, rt):
    net, N = tiny
    b = 64 if rt == 34 else 3
    M = b * rt
    g = torch.Generator(device="cuda").manual_seed(rt)
    qv = torch.randn(M, 2 * HD, generator=g, device="cuda")
    k = torch.randn(M, HD, generator=g, device="cuda")
    dO = torch.randn(M, HD, generator=g, device="cuda")
    freqs = net._w("mid_attn.fn.fn.rotary_emb.freqs")
    P = _nan(b, HEADS, rt, rt)
    O32, Ob = _nan(M, HD), _nan(M, HD, dtype=torch.bfloat16)
    N.call("dq_attn_core_fwd", qv, k, freqs, P, O32, Ob, b, rt)
    dqv, dqvb, dk = _nan(M, 2 * HD), _nan(M, 2 * HD, dtype=torch.bfloat16), _nan(M, HD)
    N.call("dq_attn_core_bwd", qv, k, freqs, P, dO, dqv, dqvb, dk, b, rt)
    torch.cuda.synchronize()

    hd = lambda x: x.double().reshape(b, rt, HEADS, 32).permute(0, 2, 1, 3)   # (b, h, n, 32)
    q_, v_, k_ = hd(qv[:, :HD]).requires_grad_(True), hd(qv[:, HD:]).requires_grad_(True), hd(k).requires_grad_(True)
    scale = 32 ** -0.5
    qr, kr = _rope64(q_, freqs), _rope64(k_, freqs)
    Pr = torch.softmax(qr @ kr.transpose(-1, -2) * scale, dim=-1)
    Or = Pr @ v_
    Or.backward(hd(dO))
    flat = lambda x: x.permute(0, 2, 1, 3).reshape(M, HD)

    with torch.no_grad():
        # score error: 32-term dot + rounding of the rotation, whose angle n * freqs carries an absolute error of
        # u * n * freqs -> delta_s <= u (40 + 2 max angle) |q||k| scale; P then carries a relative error of 2 delta_s
        # (its own score and the row's normaliser) + the __expf ulp bound at the largest |s - max| + rt (row sum) + 6
        qm, km = _rope_mag(q_), _rope_mag(k_)
        Sm = (qm @ km.transpose(-1, -2)) * scale
        s = (qr @ kr.transpose(-1, -2)) * scale
        rng = s.amax(-1, keepdim=True) - s.amin(-1, keepdim=True)
        max_ang = (rt - 1) * float(freqs.max())
        ds = U * (40 + 2 * max_ang) * Sm.amax(-1, keepdim=True)
        eps = 2 * ds + U * (_exp_ulp(rng) + rt + 6)                       # (b, h, rt, 1): relative error of P rows
        b_P = 2 * eps * Pr
        cO = 2 * eps + U * (rt + 2)
        b_O = flat(cO * (Pr @ v_.abs()))
        b_dv = flat((Pr * cO).transpose(-1, -2) @ hd(dO).abs())
        dPm = hd(dO).abs() @ v_.abs().transpose(-1, -2)
        dSm = Pr * (dPm + (Pr * dPm).sum(-1, keepdim=True))
        cS = 4 * eps.amax(-2, keepdim=True) + U * (2 * rt + 80 + 4 * max_ang)
        b_dq = flat(cS * _rope_mag(scale * dSm @ km))
        b_dk = flat(cS * _rope_mag(scale * dSm.transpose(-1, -2) @ qm))
    tag = f"attn_core b={b} rt={rt}"
    _check(tag + " P", P, Pr.detach(), b_P)
    Od = flat(Or.detach())
    _check(tag + " O f32", O32, Od, b_O)
    _check(tag + " O bf16", Ob, Od, b_O + UB * (Od.abs() + b_O))
    R_dqv = torch.cat((flat(q_.grad), flat(v_.grad)), dim=1)
    b_dqv = torch.cat((b_dq, b_dv), dim=1)
    _check(tag + " dqv", dqv, R_dqv, b_dqv)
    _check(tag + " dqv bf16", dqvb, R_dqv, b_dqv + UB * (R_dqv.abs() + b_dqv))
    _check(tag + " dk", dk, flat(k_.grad), b_dk)


def _attn_smem(rt, bwd):
    """Dynamic shared memory of attn_core_fwd / attn_core_bwd (csrc/mid.cu): q, k, v (+ dO) tiles of rt x 33 floats
    and one (two) rt x rt score tiles."""
    return 4 * ((4 if bwd else 3) * rt * 33 + (2 if bwd else 1) * rt * rt)


@pytest.mark.parametrize("bwd", [False, True])
def test_attn_core_rejects_rt_beyond_shared_memory(tiny, bwd):
    """The first rt whose tiles exceed the device's opt-in shared memory returns -2 before any launch (rt = 141 for
    the backward on sm_100a, 197 for the forward); the rt below it runs."""
    net, N = tiny
    limit = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    rt = 1
    while _attn_smem(rt, bwd) <= limit:
        rt += 1
    if bwd:
        assert rt == 141 or limit != 232448, rt
    b = 1
    freqs = net._w("mid_attn.fn.fn.rotary_emb.freqs")
    for r, want in ((rt, -2), (rt - 1, 0)):
        M = b * r
        qv, k, dO = torch.zeros(M, 2 * HD, device="cuda"), torch.zeros(M, HD, device="cuda"), torch.zeros(M, HD, device="cuda")
        P, O = _nan(b, HEADS, r, r), _nan(M, HD)
        dqv, dk = _nan(M, 2 * HD), _nan(M, HD)
        if bwd:
            P.fill_(1.0 / r)
            rc = N.call("dq_attn_core_bwd", qv, k, freqs, P, dO, dqv, None, dk, b, r, allow=(-2,))
            outs = (dqv, dk)
        else:
            rc = N.call("dq_attn_core_fwd", qv, k, freqs, P, O, None, b, r, allow=(-2,))
            outs = (P, O)
        torch.cuda.synchronize()
        assert rc == want, (r, rc)
        for o in outs:   # rejected: nothing written; accepted: everything written
            assert (torch.isnan(o).all() if want else torch.isfinite(o).all()), (r, want)


@pytest.mark.parametrize("rows,cols", [(2189, 10000), (77, 1030), (63, 300)])
def test_colsum_accumulates_against_float64(tiny, rows, cols):
    _, N = tiny
    g = torch.Generator(device="cuda").manual_seed(rows)
    x = torch.randn(rows, cols, generator=g, device="cuda")
    out0 = torch.randn(cols, generator=g, device="cuda")
    out = out0.clone()
    N.call("dq_colsum", x, out, rows, cols)
    R = out0.double() + x.double().sum(0)
    # 64 rows serially per block, then one atomic add per block onto `out`
    depth = 64 + (rows + 63) // 64 + 1
    _check(f"colsum {rows}x{cols}", out, R, depth * U * (x.double().abs().sum(0) + out0.double().abs()))


@pytest.mark.parametrize("b,rt,Nch", [(64, 34, 10000), (3, 5, 1030)])
@pytest.mark.parametrize("pad", [0, 1])
def test_mid_pack_bit_exact(tiny, b, rt, Nch, pad):
    _, N = tiny
    g = torch.Generator(device="cuda").manual_seed(b + pad)
    x = torch.randn(b * rt, Nch, generator=g, device="cuda") * 100
    out = _nan(b * (rt + 2 * pad), Nch, dtype=torch.bfloat16)
    N.call("dq_mid_pack", x, out, b, rt, Nch, pad)
    o = out.view(b, rt + 2 * pad, Nch)
    assert torch.equal(o[:, pad:pad + rt].reshape(b * rt, Nch).view(torch.int16), x.bfloat16().view(torch.int16))
    if pad:
        assert (o[:, 0].view(torch.int16) == 0).all() and (o[:, rt + 1].view(torch.int16) == 0).all()


def test_mid_pack_rejects_misaligned_pointers(tiny):
    _, N = tiny
    b, rt, Nch = 2, 3, 64
    x = torch.randn(b * rt * Nch + 2, device="cuda")
    out = _nan(b * rt * Nch + 2, dtype=torch.bfloat16)
    assert x.data_ptr() % 16 == 0 and out.data_ptr() % 16 == 0
    assert N.call("dq_mid_pack", x.data_ptr() + 4, out, b, rt, Nch, 0, allow=(-4,)) == -4
    assert N.call("dq_mid_pack", x, out.data_ptr() + 2, b, rt, Nch, 0, allow=(-4,)) == -4
    torch.cuda.synchronize()
    assert torch.isnan(out.float()).all()
    # the aligned 8-byte offset view is accepted
    N.call("dq_mid_pack", x.data_ptr() + 8, out, b, rt, Nch, 0)
    assert torch.equal(out[:b * rt * Nch].view(torch.int16), x[2:].bfloat16().view(torch.int16))


@pytest.mark.parametrize("rows", [2, 68, 2176, 8704])
@pytest.mark.parametrize("fin", [1, 8, 32])
def test_linear_fwd_bwd_against_float64(tiny, rows, fin):
    """dq_linear_bwd splits the rows over blockIdx.y (atomic partial sums) when there are >= 256 rows and fewer than
    148 column blocks: rows 2176 and 8704 take that path, rows 2 and 68 the unsplit one."""
    _, N = tiny
    fout = 128
    g = torch.Generator(device="cuda").manual_seed(rows * 7 + fin)
    x = torch.randn(rows, fin, generator=g, device="cuda")
    W = torch.randn(fout, fin, generator=g, device="cuda") / math.sqrt(fin)
    bias = torch.randn(fout, generator=g, device="cuda")
    dy = torch.randn(rows, fout, generator=g, device="cuda")
    y = _nan(rows, fout)
    N.call("dq_linear_fwd", x, W, bias, y, rows, fin, fout)
    xd, Wd, dyd = x.double(), W.double(), dy.double()
    _check(f"linear_fwd rows={rows} in={fin}", y, xd @ Wd.T + bias.double(),
           (fin + 2) * U * (xd.abs() @ Wd.abs().T + bias.double().abs()))
    dW0 = torch.randn(fout, fin, generator=g, device="cuda")
    db0 = torch.randn(fout, generator=g, device="cuda")
    dW, db, dx = dW0.clone(), db0.clone(), _nan(rows, fin)
    N.call("dq_linear_bwd", x, W, dy, dx, dW, db, rows, fin, fout)
    # worst case: every row summed serially onto the start value (covers any split / atomic order)
    _check(f"linear_bwd dW rows={rows} in={fin}", dW, dW0.double() + dyd.T @ xd,
           (rows + 2) * U * (dyd.abs().T @ xd.abs() + dW0.double().abs()))
    _check(f"linear_bwd db rows={rows} in={fin}", db, db0.double() + dyd.sum(0),
           (rows + 2) * U * (dyd.abs().sum(0) + db0.double().abs()))
    _check(f"linear_bwd dx rows={rows} in={fin}", dx, dyd @ Wd, (fout + 2) * U * (dyd.abs() @ Wd.abs()))


def test_linear_bwd_rejects_more_than_32_inputs(tiny):
    _, N = tiny
    rows, fin, fout = 4, 33, 8
    x, W, dy = torch.zeros(rows, fin, device="cuda"), torch.zeros(fout, fin, device="cuda"), torch.zeros(rows, fout, device="cuda")
    dx, dW = _nan(rows, fin), _nan(fout, fin)
    assert N.call("dq_linear_bwd", x, W, dy, dx, dW, None, rows, fin, fout, allow=(-3,)) == -3
    torch.cuda.synchronize()
    assert torch.isnan(dx).all() and torch.isnan(dW).all()


@pytest.mark.parametrize("dim", [4, 32])
def test_time_embed_against_float64(tiny, dim):
    _, N = tiny
    t = torch.tensor([0, 1, 500, 999], dtype=torch.long, device="cuda")
    b, half = t.numel(), dim // 2
    neg_e = float(torch.tensor(-(math.log(10000) / (half - 1)), dtype=torch.float32))
    out = _nan(b, dim)
    N.call("dq_time_embed", t, out, b, dim, neg_e)
    kf = torch.arange(half, dtype=torch.float64, device="cuda")
    # the kernel forms k * neg_e in fp32 (one rounding), expf (<= 2 ulp), t * f (one rounding): the angle carries a
    # relative error of u (4 + |k neg_e|); sinf / cosf add <= 2 ulp of a value <= 1
    f = torch.exp(kf * neg_e)
    a = t.double()[:, None] * f[None]
    R = torch.cat((a.sin(), a.cos()), dim=1)
    ba = U * a.abs() * (4 + (kf * neg_e).abs())[None]
    _check(f"time_embed dim={dim}", out, R, torch.cat((ba, ba), dim=1) * 2 + 4 * U)


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


@pytest.mark.parametrize("act", [0, 1, 2, 3])
def test_act_fwd_bwd_against_float64(tiny, act):
    _, N = tiny
    sp = torch.tensor([0.0, -0.0, 20.0, -20.0, 88.0, -88.0, 1e-30, -1e-30, -1.2785], device="cuda")
    z32 = torch.cat((torch.linspace(-88, 88, 20001, device="cuda"), sp, torch.nextafter(sp[2:6], torch.zeros(4, device="cuda")),
                     torch.nextafter(sp[2:6], 1e3 * sp[2:6])))
    g = torch.Generator(device="cuda").manual_seed(act)
    dy = torch.randn(z32.shape, generator=g, device="cuda")
    n = z32.numel()
    y, dx = _nan(n), _nan(n)
    N.call("dq_act_fwd", z32, y, act, n)
    N.call("dq_act_bwd", dy, z32, dx, act, n)
    z = z32.double()
    Ry, Rd = _act_ref(z, act)
    by, bd = _act_bounds(z, act)
    tiny_abs = 4 * 2.0 ** -149     # fp32 denormal spacing (softplus / SiLU tails)
    _check(f"act_fwd {act}", y, Ry, by + U * Ry.abs() + tiny_abs)
    _check(f"act_bwd {act}", dx, dy.double() * Rd, dy.double().abs() * (bd + U * Rd.abs()) + tiny_abs)


def test_fill(tiny):
    _, N = tiny
    x = _nan(1001)
    N.call("dq_fill", x, 2.5, 1001)
    assert torch.equal(x, torch.full_like(x, 2.5))


# ---------------------------------------------------------------------------------------------- 3. composed mid stage
def _per_sample(tag, got, ref, b):
    """Each sample's output within 2e-2 of that sample's maximum, cosine >= 0.999."""
    got = got.double().reshape(b, -1)
    ref = ref.double().reshape(b, -1)
    err = (got - ref).abs().amax(1)
    scale = ref.abs().amax(1)
    cos = F.cosine_similarity(got, ref, dim=1)
    worst = int((err / scale).argmax())
    print(f"PER_SAMPLE {tag}: max err / max|ref| = {float((err / scale).max()):.3g} (sample {worst}), "
          f"min cosine = {float(cos.min()):.6f}")
    assert bool((err <= 2e-2 * scale).all()), (tag, worst, float((err / scale).max()))
    assert bool((cos >= 0.999).all()), (tag, int(cos.argmin()), float(cos.min()))


def _whole(tag, got, ref):
    got, ref = got.double().flatten(), ref.double().flatten()
    e = float((got - ref).abs().max() / ref.abs().max())
    cos = float(F.cosine_similarity(got, ref, dim=0))
    print(f"PARAM_GRAD {tag}: rel {e:.3g}, cosine {cos:.6f}")
    assert e < 2e-2 and cos >= 0.999, (tag, e, cos)


def _mid_inputs(net, b, rt, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    Nm = net.mid_channels
    X = torch.randn(b * rt, Nm, generator=g, device="cuda")
    dOut = torch.randn(b * rt, Nm, generator=g, device="cuda")
    cond = torch.randn(b, 8, rt, generator=g, device="cuda")
    t = torch.randint(0, 1000, (b,), generator=g, device="cuda")
    return X, dOut, cond, t


def _run_mid(net, b, rt, X, dOut, cond, t):
    """mid block 1 and mid attention forward + backward; returns (outputs, input gradients, parameter grads, dSS)."""
    net._ensure_grads()
    net._gflat.zero_()
    net._time_path_fwd(t, b, False)
    net._dSS = torch.zeros(b, net.ss_total, device="cuda")
    cond_nlc = cond.permute(0, 2, 1).reshape(b * rt, 8).contiguous()
    out1, s1 = net._mid_block_fwd("mid_block1", X, b, rt, True)
    dX1 = net._mid_block_bwd("mid_block1", s1, dOut, b, rt)
    out2, s2 = net._mid_attn_fwd(X, cond_nlc, b, rt, True)
    dX2, dcond = net._mid_attn_bwd(s2, dOut, b, rt)
    torch.cuda.synchronize()
    grads = {k: p.grad.clone() for k, p in net._params.items()
             if k.startswith("mid_block1.") or (k.startswith("mid_attn.") and not k.endswith("freqs"))}
    return dict(out1=out1, dX1=dX1, out2=out2, dX2=dX2, dcond=dcond), grads, net._dSS.clone(), net._SS.clone()


def test_mid_block_and_attention_per_sample_at_training_batch(big):
    """_mid_block_fwd/_bwd and _mid_attn_fwd/_bwd at b = 64, rt = 34 against the oracle's blocks in float64 on the
    GPU, sample by sample; parameter gradients including the block's scale/shift (mlp.1) through _dSS."""
    import dquartic_oracle as O
    net, N = big
    b, rt = 64, 34
    Nm = net.mid_channels
    X, dOut, cond, t = _mid_inputs(net, b, rt, 21)
    outs, grads, dSS, SS = _run_mid(net, b, rt, X, dOut, cond, t)
    assert N.gemm_last_error() == 0
    sso = net.ss_off["mid_block1.mlp.1"]
    P = {k: p.detach().double().clone().requires_grad_(not k.endswith("freqs")) for k, p in net._params.items()
         if k.startswith("mid_block1.") or k.startswith("mid_attn.")}
    xin = X.double().view(b, rt, Nm).permute(0, 2, 1).requires_grad_(True)
    dO = dOut.double().view(b, rt, Nm).permute(0, 2, 1)
    with torch.backends.cudnn.flags(enabled=False):
        ss = SS[:, sso:sso + 2 * Nm].double().requires_grad_(True)
        scale, shift = ss[:, :Nm, None], ss[:, Nm:, None]
        h = O.block(P, "mid_block1.block1", xin, (scale, shift))
        ref1 = O.block(P, "mid_block1.block2", h) + xin
        ref1.backward(dO)
    to_rows = lambda y: y.permute(0, 2, 1).reshape(b * rt, Nm)
    _per_sample("mid_block1 out", outs["out1"], to_rows(ref1.detach()), b)
    _per_sample("mid_block1 dX", outs["dX1"], to_rows(xin.grad), b)
    _per_sample("mid_block1 dscale/dshift (mlp.1 via _dSS)", dSS[:, sso:sso + 2 * Nm], ss.grad, b)
    for k in ("block1.proj.weight", "block1.proj.bias", "block1.norm.g", "block2.proj.weight", "block2.proj.bias",
              "block2.norm.g"):
        _whole("mid_block1." + k, grads["mid_block1." + k], P["mid_block1." + k].grad)
    del ref1, h
    xin2 = X.double().view(b, rt, Nm).permute(0, 2, 1).requires_grad_(True)
    cd = cond.double().requires_grad_(True)
    with torch.backends.cudnn.flags(enabled=False):
        ref2 = O.mid_attention(P, xin2, cd)
        ref2.backward(dO)
    _per_sample("mid_attn out", outs["out2"], to_rows(ref2.detach()), b)
    _per_sample("mid_attn branch (out - X)", outs["out2"] - X, to_rows(ref2.detach()) - X.double(), b)
    _per_sample("mid_attn dX", outs["dX2"], to_rows(xin2.grad), b)
    _per_sample("mid_attn dcond", outs["dcond"].view(b, rt, 8).permute(0, 2, 1), cd.grad, b)
    for k in ("fn.norm.g", "fn.fn.to_qv.weight", "fn.fn.to_k.weight", "fn.fn.to_out.weight", "fn.fn.to_out.bias"):
        _whole("mid_attn." + k, grads["mid_attn." + k], P["mid_attn." + k].grad)


# ---------------------------------------------------------------------------------------------- 4. uninitialised memory
def _close(tag, a, b, rel=1e-5):
    assert torch.isfinite(a).all(), tag
    e = float((a.double() - b.double()).abs().max())
    assert e <= rel * float(b.double().abs().max()) + 1e-30, (tag, e)


def test_results_do_not_depend_on_uninitialised_memory(big, monkeypatch):
    """Every buffer UNet1d._empty hands out is filled with NaN: a TINY train step and the 10000-channel mid stage at
    b = 64 must stay finite and match the unpoisoned run (atomics reorder sums: 1e-5 relative, not bit-equal)."""
    from dquartic.model.model import DDIMDiffusionModel
    from dquartic.model.unet1d import UNet1d
    import dquartic_oracle as O

    def train_step(poison):
        if poison:
            monkeypatch.setattr(UNet1d, "_empty", lambda self, *shape, dtype=torch.float32:
                                torch.full(shape, NAN, dtype=dtype, device=self._flat.device))
        try:
            net, _ = make_net()
            d = DDIMDiffusionModel(net, device="cuda")
            b, rt, mz = 8, 34, 320
            x0 = O.det_tensor("nan_x0", (b, rt, mz)).abs().clamp(max=1)
            c2 = O.det_tensor("nan_c2", (b, rt, mz)).abs().clamp(max=1)
            c1 = torch.sigmoid(O.det_tensor("nan_c1", (b, rt)))
            noise = O.det_tensor("nan_noise", (b, rt, mz))
            t = torch.tensor([3, 90, 250, 400, 512, 700, 850, 999])
            net.train()
            loss = d.train_step(x0.cuda(), c2.cuda(), c1.cuda(), noise=noise.cuda(), t=t.cuda())
            loss.mean().backward()
            torch.cuda.synchronize()
            return loss.detach().clone(), net.flat_grads().clone()
        finally:
            monkeypatch.undo()

    l0, g0 = train_step(False)
    l1, g1 = train_step(True)
    _close("tiny loss", l1, l0)
    _close("tiny grads", g1, g0)

    net, _ = big
    b, rt = 64, 34
    inputs = _mid_inputs(net, b, rt, 33)
    ref = _run_mid(net, b, rt, *inputs)
    _nan_empty(net)
    try:
        got = _run_mid(net, b, rt, *inputs)
    finally:
        _restore_empty(net)
    for k in ref[0]:
        _close("mid " + k, got[0][k], ref[0][k])
    for k in ref[1]:
        _close("mid grad " + k, got[1][k], ref[1][k])
    _close("mid dSS", got[2], ref[2])
