"""GPU: the down- and up-path convolution kernels element by element at the shapes training runs (micro-batch 64,
RT 34: R = 2176 rows at L = 40000, 20000, .., 625), against float64 references computed on the GPU from the oracle's
blocks (cuDNN off).

Every ResnetBlock, Downsample, Upsample, the init / final convs and the attn_cond_proj path run through the same UNet1d
methods and flags a training step uses.  The kernels run once at full shape; the reference runs in chunks of samples
(activations and data gradients are compared chunk by chunk, parameter gradients are accumulated in float64).

Bounds are first-order error bounds from the kernels' arithmetic (u = 2^-24; TF32 operands carry 2^-11): a sum of
fp32 terms is bounded by (its depth) * u * (sum of |terms|), the depth counted from the launch geometry (the longest
per-thread chain over a CTA's tiles, the shared-memory / warp / block combine and the global atomics onto an element).
Gradient buffers and d scale / d shift are pre-filled with random values that must be added exactly once; every other
output is pre-filled with NaN.  `pytest -s` prints the worst err / bound of every check."""
import math

import pytest
import torch
import torch.nn.functional as F

from _util import NAN, U, _act_bounds, _act_ref, _check, _misaligned, _nan, _nan_empty, _restore_empty

pytestmark = pytest.mark.gpu

T32 = 2.0 ** -11          # unit roundoff of a TF32 operand (cvt.rna, or cf_rtf's + half ulp then truncate)
B, RT = 64, 34
CHUNK_POS = 6_000_000     # rows * L of one float64 reference chunk


# ---------------------------------------------------------------------------------------------- network and layers
@pytest.fixture(scope="module")
def net():
    """The default network at downsample_dim = 40000 (mid channels 10000); norm gains perturbed away from 1."""
    from dquartic import _native as N
    from dquartic.model.unet1d import UNet1d
    torch.cuda.manual_seed(4321)
    n = UNet1d(dim=4, channels=1, dim_mults=(1, 2, 2, 3, 3, 4, 4), conditional=True, init_cond_channels=1,
               attn_cond_channels=1, downsample_dim=40000, simple=True, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(98)
    with torch.no_grad():
        for name in n.specs:
            if name.endswith(".g"):
                w = n._w(name)
                w.copy_(1 + 0.3 * torch.randn(w.shape, generator=g, device="cuda"))
    n.mark_params_modified()
    n._ensure_grads()
    n.N = N
    yield n
    torch.cuda.synchronize()
    print(f"MEMORY max_memory_allocated = {torch.cuda.max_memory_allocated() / 2 ** 30:.1f} GiB")


def _layers(n_levels=7, L0=40000, dims=(4, 4, 8, 8, 12, 12, 16, 16)):
    """(name, L) of every ResnetBlock and resampling conv, from the default network's spec (built without a device)."""
    from dquartic.model.unet1d import param_specs
    specs = param_specs(dims[0], tuple(m // dims[0] for m in dims[1:]), 1, 1, 1, L0)
    in_out = list(zip(dims[:-1], dims[1:]))
    n = len(in_out)
    blocks, convs = [], []
    for i in range(n):
        L = L0 >> i
        blocks += [(f"downs.{i}.0", L), (f"downs.{i}.1", L)]
        convs.append((f"downs.{i}.3", L, "down" if i < n - 1 else "k3"))
    for j in range(n):
        L = L0 >> (n - 1 - j)
        blocks += [(f"ups.{j}.0", L), (f"ups.{j}.1", L)]
        convs.append((f"ups.{j}.3.1", L, "up") if j < n - 1 else (f"ups.{j}.3", L, "k3"))
    blocks.append(("final_res_block", L0))
    convs.append(("final_conv", L0, "k1"))
    assert all(p + ".block1.proj.weight" in specs for p, _ in blocks)
    assert all(p + ".weight" in specs for p, _, _ in convs)
    return blocks, convs


BLOCKS, CONVS = _layers()


def _geometry(net, pre):
    cout, cin, _ = net.specs[pre + ".block1.proj.weight"]
    has_res = (pre + ".res_conv.weight") in net.specs
    c1, c2 = (cout, cin - cout) if has_res else (cin, 0)
    return c1, c2, cout, has_res


def _samples_per_chunk(rt, L):
    return max(1, CHUNK_POS // (rt * L))


# ---------------------------------------------------------------------------------------------- launch geometry
def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _tiles(R, L, TL):
    """(total tiles, longest per-CTA tile range, most CTAs): the persistent launchers give each CTA a contiguous range
    of ceil(tiles / grid) tiles, grid = min(tiles, SMs * resident CTAs); 1 to 16 resident CTAs of 128 threads."""
    tiles = R * -(-L // TL)
    return tiles, -(-tiles // _sms()), min(tiles, 16 * _sms())


def _depth_w(R, L, TL, cin, mma):
    """Weight gradient: FFMA - thread (ci, segment) chains SL = TL / (128 / cin) positions per tile, then nseg shared
    atomics and one global atomic per CTA; MMA - each warp chains TL / 32 m16n8k8 products per tile (<= 9 additions
    each, the tensor core's accumulation counted at 2u), then 4 shared and the global atomics."""
    _, tpc, grid = _tiles(R, L, TL)
    if mma:
        return 2 * (9 * -(-TL // 32) * tpc + 4) + grid + 2
    nseg = max(1, 128 // cin)
    sl = (-(-TL // nseg) + 3) // 4 * 4
    return tpc * sl + nseg + grid + 2


def _depth_sum(R, L, TL, P, per_elem_ctas=None):
    """Bias / d g (all samples) or, with per_elem_ctas, one sample's d scale / d shift: P positions per thread and tile,
    a warp shuffle (5), the 4-warp combine and one atomic per CTA."""
    _, tpc, grid = _tiles(R, L, TL)
    return tpc * P + tpc + 5 + 4 + (grid if per_elem_ctas is None else per_elem_ctas) + 3


# ---------------------------------------------------------------------------------------------- error propagation
def _epi_fwd(u, du, g, sc1, sh, C):
    """h = SiLU(RMSNorm(u) * sc1 + sh) in float64 and a bound on |h_kernel - h| given |u_kernel - u| <= du:
    inv = rsqrt.approx(sum u^2) (<= 2^-22.9 relative, the sum C roundings); z = fma(u inv, g sqrt(C) sc1, sh);
    SiLU = z * rcp.approx(1 + ex2.approx(-log2(e) z)) (relative error <= (2 |z| + 8) u, |SiLU'| <= 1.1)."""
    nrm = u.norm(dim=1, keepdim=True).clamp_min(1e-12)
    inv = 1.0 / nrm
    uh = u * inv
    gs = g * math.sqrt(C) * sc1
    z = uh * gs + sh
    h = F.silu(z)
    e_inv = inv * (uh.abs() * du).sum(1, keepdim=True) + (C + 4) * U
    duh = du * inv + uh.abs() * (e_inv + U)
    dz = gs.abs() * duh + 5 * U * (uh * gs).abs() + U * z.abs()
    dh = 1.1 * dz + h.abs() * (2 * z.abs() + 8) * U
    return h, dh


def _epi_mag(m, u, g, sc1, sh, C):
    """Magnitude chain of the epilogue backward for |dy| <= m: returns (|du|, |d g| terms, |d scale| terms,
    |d shift| terms, per-position rounding factor of du)."""
    nrm = u.norm(dim=1, keepdim=True).clamp_min(1e-12)
    inv = 1.0 / nrm
    uh = u * inv
    n = uh * g * math.sqrt(C)
    z = n * sc1 + sh
    s = torch.sigmoid(z)
    dzm = m * s * (1 + z.abs() * (1 + s))
    duhm = dzm * (sc1 * g).abs() * math.sqrt(C)
    dotm = (duhm * uh.abs()).sum(1, keepdim=True)
    dum = inv * (duhm + uh.abs() * dotm)
    # du: s2 (C), rsqrt, u-hat, the gain product (3), SiLU' (2 |z| + 8 with ex2 / rcp), d * gs, the dot (C), (.. - ..) inv
    c_du = (2 * C + 32 + 2 * z.abs().amax(1, keepdim=True)) * U
    return dum, dzm * (sc1 * uh).abs() * math.sqrt(C), dzm * n.abs(), dzm, c_du


def _absconv(x, W, b, pad, dy=None, stride=1):
    """sum |W| |x| (+ |b|) forward, and with dy: the magnitudes (sum |W| |dy|, sum |dy| |x|, sum |dy|) of the three
    gradients of the same convolution."""
    with torch.enable_grad():
        xa = x.detach().abs().requires_grad_(dy is not None)
        Wa = W.detach().abs().requires_grad_(dy is not None)
        ba = b.detach().abs().requires_grad_(dy is not None) if b is not None else None
        y = F.conv1d(xa, Wa, ba, stride=stride, padding=pad)
        if dy is None:
            return y.detach()
        y.backward(dy)
    return xa.grad, Wa.grad, (ba.grad if ba is not None else None)


def _leaf(t):
    return t.detach().double().clone().requires_grad_(True)


# ---------------------------------------------------------------------------------------------- ResnetBlocks
def _fwd_mma(cout, cin, al):
    kci = (cin + 7) // 8
    pairs = {(8, 2), (12, 2), (12, 3), (16, 2), (16, 4)} if al else {(12, 2), (12, 3), (16, 2), (16, 4)}
    return cout >= 8 and (cout, kci) in pairs


def _bwd_variant(C, cin, al, res):
    """(MMA?, P) of the dq_conv_bwd_fused(_res) variant dispatch_fused picks for a block's conv3 + epilogue."""
    if res:
        return (False, 4) if C == 4 else (True, 2 if C == 8 else 1)
    if C == 4:
        return False, 4
    if C == 8:
        return (True, 2) if al else (False, 2)
    return True, (2 if (C == 12 and al) else 1)


def _run_block(net, pre, b, rt, L, seed):
    """Kernel forward + backward of one ResnetBlock exactly as the training step issues them; returns everything the
    reference needs (inputs, pre-filled accumulators, kernel outputs)."""
    c1, c2, C, has_res = _geometry(net, pre)
    R = b * rt
    g = torch.Generator(device="cuda").manual_seed(seed)
    x1 = torch.randn(R, c1, L, generator=g, device="cuda") + 0.25
    x2 = torch.randn(R, c2, L, generator=g, device="cuda") + 0.25 if c2 else None
    net._SS = 0.5 * torch.randn(b, net.ss_total, generator=g, device="cuda")
    dout = torch.randn(R, C, L, generator=g, device="cuda") + 0.25
    # identity-skip blocks accumulate the skip gradient into dx (downs.i.1: dskip_a; downs.0.0: dx0), as _backward_impl
    acc = (not has_res) and (pre.endswith(".1") or pre == "downs.0.0")
    old = torch.randn(R, c1, L, generator=g, device="cuda") if acc else None
    net._gflat.normal_(generator=g)
    gflat0 = net._gflat.clone()
    net._dSS = torch.randn(b, net.ss_total, generator=g, device="cuda")
    dSS0 = net._dSS.clone()
    _nan_empty(net)
    try:
        out, saved = net._resnet_fwd(pre, x1, x2, rt, True)
        dx1, dx2 = net._resnet_bwd(pre, saved, dout, rt, dx_acc=old.clone() if acc else None)
    finally:
        _restore_empty(net)
    torch.cuda.synchronize()
    _, _, u1, h1, u2 = saved
    return dict(x1=x1, x2=x2, dout=dout, old=old, gflat0=gflat0, dSS0=dSS0, out=out, u1=u1, h1=h1, u2=u2, dx1=dx1,
                dx2=dx2, dSS=net._dSS.clone(), SS=net._SS, c1=c1, c2=c2, C=C, has_res=has_res)


def _check_untouched(net, gflat0, names, dSS, dSS0, col, width):
    """Gradient-buffer ranges of other parameters and _dSS columns of other producers keep their pre-filled values."""
    spans = sorted((net.offsets[n], net.offsets[n] + math.prod(net.specs[n])) for n in names)
    lo = 0
    for a, e in spans:
        assert torch.equal(net._gflat[lo:a], gflat0[lo:a]), f"gradient buffer written in [{lo}, {a})"
        lo = e
    assert torch.equal(net._gflat[lo:], gflat0[lo:]), f"gradient buffer written beyond {lo}"
    if dSS is not None:
        assert torch.equal(dSS[:, :col], dSS0[:, :col]) and torch.equal(dSS[:, col + width:], dSS0[:, col + width:])


def _block_case(net, pre, b, rt, L, seed):
    import dquartic_oracle as O
    K = _run_block(net, pre, b, rt, L, seed)
    c1, c2, C, has_res = K["c1"], K["c2"], K["C"], K["has_res"]
    cin, R = c1 + c2, b * rt
    al = L % 4 == 0
    sq = math.sqrt(C)
    tag = f"{pre} b={b} rt={rt} L={L}"
    names = [pre + s for s in (".block1.proj.weight", ".block1.proj.bias", ".block1.norm.g", ".block2.proj.weight",
                               ".block2.proj.bias", ".block2.norm.g")]
    if has_res:
        names += [pre + ".res_conv.weight", pre + ".res_conv.bias"]
    P = {n: _leaf(net._w(n).view(net.specs[n])) for n in names}
    W1, b1, g1 = P[names[0]], P[names[1]], P[names[2]]
    W2, b2, g2 = P[names[3]], P[names[4]], P[names[5]]
    Wr, br = (P[names[6]], P[names[7]]) if has_res else (None, None)
    Od = {n: p for n, p in P.items()}
    sso = net.ss_off[pre + ".mlp.1"]
    ss = K["SS"][:, sso:sso + 2 * C].double().requires_grad_(True)        # (b, 2C): per-sample reference gradients
    fmma = _fwd_mma(C, cin, al)
    bmma2, P2 = _bwd_variant(C, C, al, False)
    bmma1, P1 = _bwd_variant(C, cin, al, has_res)
    kco = (C + 7) // 8
    # conv rounding factors (x Sum |w||x|): FFMA chains, or TF32 operands + the tensor core's accumulation
    c_f1 = (2 * T32 + 2 * U * (27 * ((cin + 7) // 8) + 4)) if fmma else (3 * cin + 3) * U
    c_f2 = (2 * T32 + 2 * U * (27 * kco + 4)) if fmma else (3 * C + 3) * U
    c_fr = (2 * T32 + 2 * U * (9 * ((cin + 7) // 8) + 4)) if fmma else (cin + 3) * U
    c_dx2 = (T32 + 2 * U * (27 * kco + 4)) if bmma2 else (3 * C + 4) * U
    c_dx1 = (T32 + 2 * U * (27 * kco + 4)) if bmma1 else (3 * C + 4) * U
    c_dxr = (2 * T32 + 2 * U * (9 * kco + 4)) if bmma1 else (C + 4) * U
    Dw2, Dw1 = _depth_w(R, L, 128 * P2, C, bmma2), _depth_w(R, L, 128 * P1, cin, bmma1)
    Db2, Db1 = _depth_sum(R, L, 128 * P2, P2), _depth_sum(R, L, 128 * P1, P1)
    Dss = _depth_sum(R, L, 128 * P1, P1, per_elem_ctas=rt * -(-L // (128 * P1)) + 1)
    acc_m = {k: torch.zeros_like(p, dtype=torch.float64) for k, p in P.items()}   # |terms| and propagated parts
    acc_p = {k: torch.zeros_like(p, dtype=torch.float64) for k, p in P.items()}
    mss = torch.zeros(b, 2 * C, dtype=torch.float64, device="cuda")
    pss = torch.zeros_like(mss)
    with torch.backends.cudnn.flags(enabled=False):
        spc = _samples_per_chunk(rt, L)
        for s0 in range(0, b, spc):
            s1 = min(b, s0 + spc)
            rows = slice(s0 * rt, s1 * rt)
            xd = K["x1"][rows].double() if not c2 else torch.cat((K["x1"][rows], K["x2"][rows]), 1).double()
            sc = ss[s0:s1, :C].repeat_interleave(rt, 0)[:, :, None]
            sh = ss[s0:s1, C:].repeat_interleave(rt, 0)[:, :, None]
            with torch.no_grad():
                # ---- forward: u1, h1 from x; u2, out from the kernel's own h1 (each stage against its own input)
                u1r = F.conv1d(xd, W1, b1, padding=1)
                du1 = c_f1 * _absconv(xd, W1, b1, 1)
                h1r, dh1 = _epi_fwd(u1r, du1, g1, sc + 1, sh, C)
                h1r_o = O.block(Od, pre + ".block1", xd, (sc, sh))
                _check(tag + " u1", K["u1"][rows], u1r, du1, rt, rows.start)
                _check(tag + " h1", K["h1"][rows], h1r_o, dh1 + U * h1r.abs(), rt, rows.start)
                h1g = K["h1"][rows].double()
                u2r = F.conv1d(h1g, W2, b2, padding=1)
                # the kernel's conv2 reads its own h1 tile (halo positions recomputed, TF32-rounded in the MMA kernel)
                du2 = c_f2 * _absconv(h1g, W2, b2, 1) + _absconv(2 * dh1 + (T32 * h1g.abs() if fmma else 0), W2, None, 1)
                h2r, dh2 = _epi_fwd(u2r, du2, g2, 1.0, 0.0, C)
                if has_res:
                    res = F.conv1d(xd, Wr, br)
                    dres = c_fr * _absconv(xd, Wr, br, 0)
                else:
                    res, dres = xd, 0
                outr = O.block(Od, pre + ".block2", h1g) + res
                _check(tag + " u2", K["u2"][rows], u2r, du2, rt, rows.start)
                _check(tag + " out", K["out"][rows], outr, dh2 + dres + 2 * U * outr.abs(), rt, rows.start)
                del u1r, du1, h1r, h1r_o, u2r, h2r, dh2, res, outr
            # ---- backward: block2 at the saved u2 / h1, block1 at the saved u1 and the reference d h1
            dout = K["dout"][rows].double()
            u2g = K["u2"][rows].double()
            h1l = h1g.clone().requires_grad_(True)
            t = F.conv1d(h1l, W2, b2, padding=1)
            F.silu(O.rmsnorm(t + (u2g - t).detach(), g2)).backward(dout)
            dh1_ref = h1l.grad
            u1g = K["u1"][rows].double()
            xl = xd.clone().requires_grad_(True)
            t = F.conv1d(xl, W1, b1, padding=1)
            h1e = F.silu(O.rmsnorm(t + (u1g - t).detach(), g1) * (sc + 1) + sh)
            resl = F.conv1d(xl, Wr, br) if has_res else xl
            ((h1e * dh1_ref).sum() + (resl * dout).sum()).backward()
            with torch.no_grad():
                # block2 magnitudes: |du2| chain, its rounding, the TF32 rounding of du in the MMA kernels
                dum2, gm2, _, _, c2el = _epi_mag(dout.abs(), u2g, g2, 1.0, 0.0, C)
                ddu2 = c2el * dum2 + (T32 * dum2 if bmma2 else 0)
                mdh1, mW2, mb2 = _absconv(h1g, W2, b2, 1, dum2)
                pdh1, pW2, pb2 = _absconv(h1g, W2, b2, 1, ddu2)
                ddh1 = pdh1 + c_dx2 * mdh1
                acc_m[names[3]] += mW2 * (Dw2 * U + (T32 if bmma2 else 0))
                acc_p[names[3]] += pW2
                acc_m[names[4]] += mb2 * Db2 * U
                acc_p[names[4]] += pb2
                acc_m[names[5]] += (gm2.sum((0, 2)) * (Db2 * U + c2el.max())).view(1, C, 1)
                # block1: the same chain fed with |d h1| (own rounding) and with the bound on d h1 (propagated)
                m1 = dh1_ref.abs() + ddh1
                dum1, gm1, scm1, shm1, c1el = _epi_mag(m1, u1g, g1, sc + 1, sh, C)
                pdum1, pgm1, pscm1, pshm1, _ = _epi_mag(ddh1, u1g, g1, sc + 1, sh, C)
                ddu1 = c1el * dum1 + pdum1 + (T32 * dum1 if bmma1 else 0)
                mdx, mW1, mb1 = _absconv(xd, W1, b1, 1, dum1)
                pdx, pW1, pb1 = _absconv(xd, W1, b1, 1, ddu1)
                acc_m[names[0]] += mW1 * (Dw1 * U + (T32 if bmma1 else 0))
                acc_p[names[0]] += pW1
                acc_m[names[1]] += mb1 * Db1 * U
                acc_p[names[1]] += pb1
                acc_m[names[2]] += (gm1.sum((0, 2)) * (Db1 * U + c1el.max())).view(1, C, 1)
                acc_p[names[2]] += pgm1.sum((0, 2)).view(1, C, 1)
                per_s = lambda v: v.view(s1 - s0, rt, C, L).sum((1, 3))
                mss[s0:s1] += torch.cat((per_s(scm1), per_s(shm1)), 1) * (Dss * U + c1el.max())
                pss[s0:s1] += torch.cat((per_s(pscm1), per_s(pshm1)), 1)
                bdx = pdx + c_dx1 * mdx
                if has_res:
                    mdxr, mWr, mbr = _absconv(xd, Wr, br, 0, dout.abs())
                    bdx = bdx + c_dxr * mdxr
                    Dwr = _depth_w(R, L, 128 * P1, cin, bmma1)
                    acc_m[names[6]] += mWr * (Dwr * U + (2 * T32 if bmma1 else 0))
                    acc_m[names[7]] += mbr * Db1 * U
                    ref_dx = xl.grad
                else:
                    ref_dx = xl.grad
                    bdx = bdx + (3 * C + 6) * U * dout.abs()     # dadd enters the FFMA chain first
                if K["old"] is not None:
                    old = K["old"][rows].double()
                    ref_dx = ref_dx.clone()
                    ref_dx[:, :c1] += old
                    bdx[:, :c1] += (3 * C + 6) * U * old.abs() + 2 * U * ref_dx[:, :c1].abs()
                bdx = bdx + U * ref_dx.abs()
                _check(tag + " dx1", K["dx1"][rows], ref_dx[:, :c1], bdx[:, :c1], rt, rows.start)
                if c2:
                    _check(tag + " dx2", K["dx2"][rows], ref_dx[:, c1:], bdx[:, c1:], rt, rows.start)
            del xl, h1l, t, h1e, resl, dh1_ref
    g0 = K["gflat0"]
    for n in names:
        lo = net.offsets[n]
        n_el = math.prod(net.specs[n])
        old = g0[lo:lo + n_el].view(net.specs[n]).double()
        got = net._gflat[lo:lo + n_el].view(net.specs[n])
        ref = old + P[n].grad
        _check(f"{tag} d {n[len(pre) + 1:]}", got, ref, acc_m[n] + acc_p[n] + 2 * U * (old.abs() + ref.abs()))
    d0 = K["dSS0"][:, sso:sso + 2 * C].double()
    _check(tag + " d scale / d shift per sample", K["dSS"][:, sso:sso + 2 * C], d0 + ss.grad,
           mss + pss + 2 * U * (d0.abs() + (d0 + ss.grad).abs()))
    _check_untouched(net, g0, names, K["dSS"], K["dSS0"], sso, 2 * C)


@pytest.mark.parametrize("pre,L", BLOCKS, ids=[p for p, _ in BLOCKS])
def test_resnet_block_per_element_at_training_shape(net, pre, L):
    """dq_resblock_fwd and the block backward (dq_conv_bwd_fused for block2, dq_conv_bwd_fused_res or dq_conv_bwd_fused
    with dadd / the skip-gradient accumulation for block1) of one ResnetBlock at b = 64, rt = 34."""
    _block_case(net, pre, B, RT, L, seed=[p for p, _ in BLOCKS].index(pre))


def test_resnet_block_at_136_rows_per_sample(net):
    """Level-0 ResnetBlock at rt = 136 (b = 16, the same 2176 rows): a sample spans four times as many tiles."""
    _block_case(net, "downs.0.1", 16, 136, 40000, seed=136)


# ---------------------------------------------------------------------------------------------- Downsample / Upsample / k3 / k1
def _plain_bwd_tile(kind, cout, L):
    """(TL, P) of the backward kernel a plain conv takes (dispatch in csrc/conv_fused.cu)."""
    if kind == "k1":
        return 512, 4                                    # conv_bwd_fused_kernel<1, 1, 4, VEC = 4>
    if kind in ("up", "down"):
        P = 4 if cout == 4 else 2
    else:
        P = {4: 4, 8: 2, 12: 2 if L % 4 == 0 else 1, 16: 1}[cout]
    return 128 * P, P


@pytest.mark.parametrize("pre,L,kind", CONVS, ids=[p for p, _, _ in CONVS])
def test_resampling_and_plain_conv_per_element_at_training_shape(net, pre, L, kind):
    """Downsample (k4 s2, dx accumulated onto the skip gradient as _backward_impl does), the last level's k3 conv, Upsample
    (nearest x2 + k3: one-pass forward and backward), the last up conv and final_conv (cout 1, K 1) at b = 64, rt = 34."""
    wname, bname = pre + ".weight", pre + ".bias"
    cout, cin, k = net.specs[wname]
    R, rt = B * RT, RT
    Lin = L
    Lout = {"down": L // 2, "up": 2 * L}.get(kind, L)
    stride, pad, up = {"down": (2, 1, 1), "up": (1, 1, 2), "k3": (1, 1, 1), "k1": (1, 0, 1)}[kind]
    acc = pre.startswith("downs.")                      # the down path adds the skip gradient (dx1 = dskip_c)
    g = torch.Generator(device="cuda").manual_seed(len(pre) * 7 + L)
    x = torch.randn(R, cin, Lin, generator=g, device="cuda") + 0.5
    dy = torch.randn(R, cout, Lout, generator=g, device="cuda") + 0.5
    old = torch.randn(R, cin, Lin, generator=g, device="cuda") if acc else None
    net._gflat.normal_(generator=g)
    gflat0 = net._gflat.clone()
    _nan_empty(net)
    try:
        y, _ = net._conv_fwd(x, None, wname, bname, k, stride, pad, up, Lout, rps=rt)
        dx, _ = net._conv_bwd(dy, x, None, wname, bname, k, stride, pad, up, dx1=old.clone() if acc else None, rps=rt)
    finally:
        _restore_empty(net)
    torch.cuda.synchronize()
    W, bias = _leaf(net._w(wname).view(cout, cin, k)), _leaf(net._w(bname))
    TL, P = _plain_bwd_tile(kind, cout, Lout)
    Dw = _depth_w(R, max(Lin, Lout), TL, cin, False)
    Db = _depth_sum(R, max(Lin, Lout), TL, P)
    taps_dx = {"down": 2 * cout, "up": 6 * cout}.get(kind, k * cout)
    mW = torch.zeros_like(W)
    mb = torch.zeros_like(bias)
    tag = f"{pre} ({kind}) L={L}"

    def graph(xin, Wt, bt):
        xu = F.interpolate(xin, scale_factor=2, mode="nearest") if kind == "up" else xin
        return F.conv1d(xu, Wt, bt, stride=stride, padding=pad)

    with torch.backends.cudnn.flags(enabled=False):
        spc = _samples_per_chunk(rt, max(Lin, Lout) * max(1, cin // 4))
        for s0 in range(0, B, spc):
            rows = slice(s0 * rt, min(B, s0 + spc) * rt)
            xl = x[rows].double().requires_grad_(True)
            yr = graph(xl, W, bias)
            yr.backward(dy[rows].double())
            with torch.no_grad():
                with torch.enable_grad():
                    xa = x[rows].double().abs().requires_grad_(True)
                    Wa = W.detach().abs().requires_grad_(True)
                    ba = bias.detach().abs().requires_grad_(True)
                    ya = graph(xa, Wa, ba)
                    ya.backward(dy[rows].double().abs())
                _check(tag + " y", y[rows], yr, (cin * k + 3) * U * ya, rt, rows.start)
                ref = xl.grad + (old[rows].double() if acc else 0)
                # the accumulated old value enters the kernel's FMA chain first: it carries the chain's roundings too
                bnd = (taps_dx + 4) * U * (xa.grad + (old[rows].double().abs() if acc else 0)) + 2 * U * ref.abs()
                _check(tag + " dx", dx[rows], ref, bnd, rt, rows.start)
                mW += Wa.grad
                mb += ba.grad
            del xl, yr, xa, ya
    for n, p, m, D in ((wname, W, mW, Dw), (bname, bias, mb, Db)):
        lo, ne = net.offsets[n], p.numel()
        o = gflat0[lo:lo + ne].view(p.shape).double()
        r = o + p.grad
        _check(f"{tag} d {n.rsplit('.', 1)[1]}", net._gflat[lo:lo + ne].view(p.shape), r, D * U * m + 2 * U * (o.abs() + r.abs()))
    _check_untouched(net, gflat0, [wname, bname], None, None, 0, 0)


# ---------------------------------------------------------------------------------------------- init_conv
def test_init_conv_forward_and_one_pass_backward_per_element(net):
    """init_conv = Conv1d(2 -> 4, k7, p3) over cat(cond * (scale + 1) + shift, x) forward (pipelined k7 kernel with the
    ConditionalScaleShift on the staged rows) and dq_initconv_bwd (dW, db, per-sample d scale / d shift) at b = 64,
    rt = 34, L = 40000."""
    N = net.N
    R, rt, L = B * RT, RT, 40000
    cout = net.specs["init_conv.weight"][0]
    g = torch.Generator(device="cuda").manual_seed(77)
    cond = torch.rand(R, 1, L, generator=g, device="cuda")
    x = torch.randn(R, 1, L, generator=g, device="cuda") + 0.5
    d = torch.randn(R, cout, L, generator=g, device="cuda") + 0.25
    net._SS = 0.5 * torch.randn(B, net.ss_total, generator=g, device="cuda")
    ico = net.ss_off["init_cond_proj.to_scale_shift.1"]
    net._gflat.normal_(generator=g)
    gflat0 = net._gflat.clone()
    dSS = torch.randn(B, net.ss_total, generator=g, device="cuda")
    dSS0 = dSS.clone()
    _nan_empty(net)
    try:
        y, _ = net._conv_fwd(cond, x, "init_conv.weight", "init_conv.bias", 7, 1, 3, 1, L, in_ss=ico, rps=rt)
    finally:
        _restore_empty(net)
    scratch = torch.zeros(B, cout // 4, 88, device="cuda")
    rc = N.call("dq_initconv_bwd", d, cond, x, net._SS[:, ico:].data_ptr(), net.ss_total, net._w("init_conv.weight"),
                net._gw("init_conv.weight"), net._gw("init_conv.bias"), dSS[:, ico:].data_ptr(), scratch, cout, R, L, rt,
                allow=(1,))
    torch.cuda.synchronize()
    assert rc == 0, "the one-pass init_conv backward must cover the training shape"
    W, bias = _leaf(net._w("init_conv.weight").view(cout, 2, 7)), _leaf(net._w("init_conv.bias"))
    ss = net._SS[:, ico:ico + 2].double().requires_grad_(True)
    # one-pass backward: per (row, chunk of L) block 4 FMAs x chunk / 512 iterations per thread + block reduce, one
    # atomic per (row, chunk) of the sample into its record, then the finalize's 3 roundings and one atomic per sample
    nchunk = -(-L // 8192)
    chunk = (-(-L // nchunk) + 511) // 512 * 512
    Dg = chunk // 128 + 9 + rt * nchunk + 2
    mW = torch.zeros_like(W)
    mb = torch.zeros_like(bias)
    mss = torch.zeros(B, 2, dtype=torch.float64, device="cuda")
    tag = f"init_conv L={L}"
    with torch.backends.cudnn.flags(enabled=False):
        spc = _samples_per_chunk(rt, L * 2)
        for s0 in range(0, B, spc):
            s1 = min(B, s0 + spc)
            rows = slice(s0 * rt, s1 * rt)
            sc1 = ss[s0:s1, 0:1].repeat_interleave(rt, 0)[:, :, None] + 1
            sh = ss[s0:s1, 1:2].repeat_interleave(rt, 0)[:, :, None]
            cd = cond[rows].double()
            inp = torch.cat((cd * sc1 + sh, x[rows].double()), 1)
            yr = F.conv1d(inp, W, bias, padding=3)
            yr.backward(d[rows].double())
            with torch.no_grad():
                ia = torch.cat((cd * sc1.abs() + sh.abs(), x[rows].double().abs()), 1)
                ma = F.conv1d(ia, W.abs(), bias.abs(), padding=3)
                _check(tag + " y", y[rows], yr, (14 + 6) * U * ma, rt, rows.start)
                da = d[rows].double().abs()
                with torch.enable_grad():
                    ial = ia.clone().requires_grad_(True)
                    Wa = W.detach().abs().requires_grad_(True)
                    ba = bias.detach().abs().requires_grad_(True)
                    F.conv1d(ial, Wa, ba, padding=3).backward(da)
                mW += Wa.grad
                mb += ba.grad
                # |d scale_s| terms: sum |cond| (|W0|^T |d|); |d shift_s|: sum |W0|^T |d|
                back = F.conv_transpose1d(da, W.detach().abs()[:, 0:1], padding=3)
                per_s = lambda v: v.view(s1 - s0, -1).sum(1)
                mss[s0:s1, 0] += per_s(back * cd.abs())
                mss[s0:s1, 1] += per_s(back)
            del inp, yr
    Dw = Dg + B + 6
    for n, p, m in (("init_conv.weight", W, mW), ("init_conv.bias", bias, mb)):
        lo, ne = net.offsets[n], p.numel()
        o = gflat0[lo:lo + ne].view(p.shape).double()
        r = o + p.grad
        _check(f"{tag} d {n.split('.')[1]}", net._gflat[lo:lo + ne].view(p.shape), r, Dw * U * m + 2 * U * (o.abs() + r.abs()))
    d0 = dSS0[:, ico:ico + 2].double()
    r = d0 + ss.grad
    _check(tag + " d scale / d shift per sample", dSS[:, ico:ico + 2], r, (Dg + 56 + 8) * U * mss + 2 * U * (d0.abs() + r.abs()))
    _check_untouched(net, gflat0, ["init_conv.weight", "init_conv.bias"], dSS, dSS0, ico, 2)


# ---------------------------------------------------------------------------------------------- attn_cond_proj
def test_attn_cond_proj_convs_and_gelu_block_backward_over_rt(net):
    """attn_cond_proj: Conv1d(1 -> 8, k7, p3) + GELU (pre-activation saved) and Conv1d(8 -> 8, k1) over rt = 34 for
    b = 64 samples, forward and backward as _forward_impl / _backward_impl issue them (dq_block_bwd for the GELU)."""
    from dquartic.model.unet1d import ACT_GELU
    R, rt = B, RT
    acd = 8
    g = torch.Generator(device="cuda").manual_seed(55)
    ac0 = torch.rand(R, 1, rt, generator=g, device="cuda")
    da2 = torch.randn(R, acd, rt, generator=g, device="cuda") + 0.25
    names = ["attn_cond_proj.1.0.weight", "attn_cond_proj.1.0.bias", "attn_cond_proj.1.2.weight", "attn_cond_proj.1.2.bias"]
    net._gflat.normal_(generator=g)
    gflat0 = net._gflat.clone()
    _nan_empty(net)
    try:
        a1, a1u = net._conv_fwd(ac0, None, names[0], names[1], 7, 1, 3, 1, rt, act=ACT_GELU, save_u=True, rps=1)
        a2, _ = net._conv_fwd(a1, None, names[2], names[3], 1, 1, 0, 1, rt, rps=1)
        da1, _ = net._conv_bwd(da2, a1, None, names[2], names[3], 1, 1, 0, 1, rps=1)
        da1u = net._block_bwd(da1, a1u, None, None, ACT_GELU, 1)
        net._conv_bwd(da1u, ac0, None, names[0], names[1], 7, 1, 3, 1, need_dx1=False, rps=1)
    finally:
        _restore_empty(net)
    torch.cuda.synchronize()
    P = {n: _leaf(net._w(n).view(net.specs[n])) for n in names}
    W0, b0, W2, b2 = (P[n] for n in names)
    with torch.backends.cudnn.flags(enabled=False):
        xd = ac0.double()
        with torch.no_grad():
            u_r = F.conv1d(xd, W0, b0, padding=3)
            _check("attn_cond conv k7 (pre-activation)", a1u, u_r, 10 * U * _absconv(xd, W0, b0, 3), 1)
            z = a1u.double()
            act, _ = _act_ref(z, 2)
            bf, bd = _act_bounds(z, 2)
            _check("attn_cond GELU", a1, act, bf + U * act.abs(), 1)
            a1g = a1.double()
            _check("attn_cond conv k1", a2, F.conv1d(a1g, W2, b2), (acd + 3) * U * _absconv(a1g, W2, b2, 0), 1)
        # backward stage by stage, each from the kernel's own input of that stage
        a1l = a1g.clone().requires_grad_(True)
        F.conv1d(a1l, W2, b2).backward(da2.double())
        with torch.no_grad():
            mdx, mW2, mb2 = _absconv(a1g, W2, b2, 0, da2.double().abs())
            _check("attn_cond conv k1 dx", da1, a1l.grad, (acd + 4) * U * mdx, 1)
            _, d_act = _act_ref(z, 2)
            r = da1.double() * d_act
            _check("attn_cond GELU backward (dq_block_bwd)", da1u, r, da1.double().abs() * (bd + U * d_act.abs()) + U * r.abs(), 1)
        xl = xd.clone().requires_grad_(True)
        F.conv1d(xl, W0, b0, padding=3).backward(da1u.double())
        with torch.no_grad():
            _, mW0, mb0 = _absconv(xd, W0, b0, 3, da1u.double().abs())
    n_terms = R * rt + 4                                 # any summation order of R * rt terms
    for n, m in zip(names, (mW0, mb0, mW2, mb2)):
        lo, ne = net.offsets[n], P[n].numel()
        o = gflat0[lo:lo + ne].view(P[n].shape).double()
        r = o + P[n].grad
        _check(f"attn_cond d {n}", net._gflat[lo:lo + ne].view(P[n].shape), r, n_terms * U * m + 2 * U * (o.abs() + r.abs()))
    _check_untouched(net, gflat0, names, None, None, 0, 0)


# ---------------------------------------------------------------------------------------------- 4-byte aligned views
ALIGN_CASES = [
    # (path, cout, c1, c2, dadd / accumulate, pointers offset in turn)
    ("k1 cout 1 (VEC = 4 kernel)", 1, 4, 0, True, ("dy", "x1", "dadd", "dx1")),
    ("k3 cout 4 bulk FFMA", 4, 4, 4, True, ("dy", "x1", "x2", "dadd", "dx1", "dx2")),
    ("k3 cout 4 bulk FFMA, no dadd / accumulate", 4, 4, 4, False, ("dy", "x1", "x2", "dx1", "dx2")),
    ("res cout 4", 4, 4, 4, False, ("dy", "u", "x1", "x2", "dx1", "dx2", "dyo")),
]


@pytest.mark.parametrize("case", ALIGN_CASES, ids=[c[0] for c in ALIGN_CASES])
def test_fused_conv_backward_accepts_4_byte_aligned_views(net, case):
    """dq_conv_bwd_fused / dq_conv_bwd_fused_res with each pointer in turn a view 4 bytes past a 16-byte boundary: the
    dispatch leaves every vector path whose accesses that pointer would break, and each result meets the float64
    reference's bound (a 4-channel res_conv case that is not covered runs the documented two-call composition)."""
    import dquartic_oracle as O
    N = net.N
    path, cout, c1, c2, with_add, ptrs = case
    res = path.startswith("res")
    K = 1 if cout == 1 else 3
    b, rt, L = 2, 5, 2048
    R, cin = b * rt, c1 + c2
    g = torch.Generator(device="cuda").manual_seed(len(path))
    W = 0.3 * torch.randn(cout, cin, K, generator=g, device="cuda")
    Wr = 0.3 * torch.randn(cout, cin, generator=g, device="cuda")
    gain = 1 + 0.3 * torch.randn(cout, generator=g, device="cuda")
    SS = 0.5 * torch.randn(b, 2 * cout, generator=g, device="cuda")
    T = dict(dy=torch.randn(R, cout, L, generator=g, device="cuda") + 0.25,
             u=torch.randn(R, cout, L, generator=g, device="cuda"),
             x1=torch.randn(R, c1, L, generator=g, device="cuda") + 0.5,
             x2=torch.randn(R, c2, L, generator=g, device="cuda") + 0.5,
             dyo=torch.randn(R, cout, L, generator=g, device="cuda"),
             dadd=torch.randn(R, c1, L, generator=g, device="cuda"))
    old1 = torch.randn(R, c1, L, generator=g, device="cuda")
    old2 = torch.randn(R, c2, L, generator=g, device="cuda")

    # float64 reference and bounds (the plain kernels: K * cout terms per dx; any order of R * L terms per dW / db)
    with torch.backends.cudnn.flags(enabled=False):
        xd = torch.cat((T["x1"], T["x2"]), 1).double().requires_grad_(True)
        Wd, Wrd = _leaf(W), _leaf(Wr)
        ssd = SS.double().requires_grad_(True)
        dy = T["dy"].double()
        if res:
            t = F.conv1d(xd, Wd, None, padding=1)
            u = T["u"].double()
            sc = ssd[:, :cout].repeat_interleave(rt, 0)[:, :, None]
            sh = ssd[:, cout:].repeat_interleave(rt, 0)[:, :, None]
            h = F.silu(O.rmsnorm(t + (u - t).detach(), gain.double().view(1, cout, 1)) * (sc + 1) + sh)
            ((h * dy).sum() + (F.conv1d(xd, Wrd[:, :, None]) * T["dyo"].double()).sum()).backward()
            with torch.no_grad():
                dum, _, _, _, cel = _epi_mag(dy.abs(), u, gain.double().view(1, cout, 1), sc + 1, sh, cout)
                mdx, mW, _ = _absconv(xd, Wd, None, 1, dum)
                pdx, pW, _ = _absconv(xd, Wd, None, 1, cel * dum)
                mdxr, mWr, _ = _absconv(xd, Wrd[:, :, None], None, 0, T["dyo"].double().abs())
                ref_dx = xd.grad
                bdx = pdx + (4 * cout + 5) * U * (mdx + mdxr) + 2 * U * ref_dx.abs()
        else:
            F.conv1d(xd, Wd, None, padding=K // 2).backward(dy)
            with torch.no_grad():
                mdx, mW, _ = _absconv(xd, Wd, None, K // 2, dy.abs())
                ref_dx = xd.grad.clone()
                bdx = (K * cout + 4) * U * mdx
                if with_add:
                    extra = torch.cat((T["dadd"] + old1, old2), 1).double()
                    ref_dx += extra
                    bdx += (K * cout + 4) * U * torch.cat((T["dadd"].abs() + old1.abs(), old2.abs()), 1).double() + 2 * U * ref_dx.abs()
                pW = 0
                bdx = bdx + U * ref_dx.abs()
    bW = (R * L + 4) * U * mW + pW + U * Wd.grad.abs()

    for which in (None,) + ptrs:
        A = {k: (_misaligned(v) if k == which else v.clone()) for k, v in T.items()}
        base1 = old1 if (with_add and not res) else None
        dx1 = _misaligned(base1) if which == "dx1" and base1 is not None else (base1.clone() if base1 is not None else None)
        if dx1 is None:
            dx1 = _misaligned(torch.full((R, c1, L), NAN, device="cuda")) if which == "dx1" else _nan(R, c1, L)
        dx2 = None
        if c2:
            base2 = old2 if (with_add and not res) else None
            dx2 = (_misaligned(base2) if base2 is not None else _misaligned(torch.full((R, c2, L), NAN, device="cuda"))) \
                if which == "dx2" else (base2.clone() if base2 is not None else _nan(R, c2, L))
        dw = torch.zeros(cout, cin, K, device="cuda")
        dwr = torch.zeros(cout, cin, device="cuda")
        db, dbr, dg = torch.zeros(cout, device="cuda"), torch.zeros(cout, device="cuda"), torch.zeros(cout, device="cuda")
        dss = torch.zeros(b, 2 * cout, device="cuda")
        if res:
            rc = N.call("dq_conv_bwd_fused_res", A["dy"], A["u"], gain, SS, 2 * cout, 1, A["x1"], c1, A["x2"], c2, W,
                        dx1, dx2, dw, db, dg, dss, A["dyo"], Wr, dwr, dbr, cout, R, L, rt, allow=(1,))
            if rc == 1:   # not covered: block1 backward, then the 1x1 conv accumulated (UNet1d._resnet_bwd)
                N.call("dq_conv_bwd_fused", A["dy"], A["u"], gain, SS, 2 * cout, 1, A["x1"], c1, A["x2"], c2, W, None,
                       dx1, 0, dx2, 0, dw, db, dg, dss, cout, 3, R, L, rt)
                N.call("dq_conv_bwd_fused", A["dyo"], None, None, None, 0, 0, A["x1"], c1, A["x2"], c2, Wr, None,
                       dx1, 1, dx2, 1, dwr, dbr, None, None, cout, 1, R, L, rt)
        else:
            N.call("dq_conv_bwd_fused", A["dy"], None, None, None, 0, 0, A["x1"], c1, A["x2"] if c2 else None, c2, W,
                   A["dadd"] if with_add else None, dx1, 1 if with_add else 0, dx2, 1 if (with_add and c2) else 0,
                   dw, db, None, None, cout, K, R, L, rt)
        torch.cuda.synchronize()
        tag = f"{path} offset {which or 'none'}"
        _check(tag + " dx1", dx1, ref_dx[:, :c1], bdx[:, :c1], rt)
        if c2:
            _check(tag + " dx2", dx2, ref_dx[:, c1:], bdx[:, c1:], rt)
        _check(tag + " dW", dw, Wd.grad, bW)
        if res:
            _check(tag + " dWres", dwr, Wrd.grad, (R * L + 4) * U * mWr.squeeze(-1) + U * Wrd.grad.abs())
