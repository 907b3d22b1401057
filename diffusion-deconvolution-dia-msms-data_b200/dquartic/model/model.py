"""`DDIMDiffusionModel` — drop-in for /root/reference/dquartic/model/model.py:151-406 on B200.

Same constructor, attributes (`betas, alphas, alpha_bars, loss_weight, normalize, unnormalize, pred_type,
ms1_loss_weight, model, num_timesteps, device`) and methods (`q_sample, p_sample, sample, train_step`).
The schedule tables are built exactly like the reference (fp64 -> fp32, fp32 cumprod) so they are bit-identical;
q_sample, the reverse step, the final un-normalise and the epsilon-MSE are single fused CUDA kernels.

Batched semantics (the reference only runs at b = 1, SURVEY.md §8c): `train_step` returns a (b,) tensor whose
entries are the batch-mean MSE times `loss_weight[t_i]`; call `.mean().backward()` (the harness does).
"""
import math

import numpy as np
import torch

from .. import _native as N
from .model_interface import ModelInterface


def get_linear_beta_schedule(num_timesteps, beta_start=0.0001, beta_end=0.02):
    return torch.linspace(beta_start, beta_end, num_timesteps, dtype=torch.float64)


def get_cosine_beta_schedule(num_timesteps, s=0.008):
    t = torch.linspace(0, num_timesteps, num_timesteps + 1, dtype=torch.float64)
    f = torch.cos(((t / num_timesteps) + s) / (1 + s) * math.pi * 0.5) ** 2
    f = f / f[0]
    return torch.clip(1 - (f[1:] / f[:-1]), 0, 0.999)


def get_alphas(betas):
    return 1.0 - betas


def get_alpha_bars(alpha):
    return torch.cumprod(alpha, dim=0)


def normalize_to_neg_one_to_one(img):
    if img.is_cuda and img.dtype == torch.float32:
        out = torch.empty_like(img, memory_format=torch.contiguous_format)
        N.call("dq_mix_affine", img.contiguous(), None, 1.0, 0.0, 2.0, -1.0, out, img.numel())
        return out
    return img * 2 - 1


def unnormalize_to_zero_to_one(t):
    if t.is_cuda and t.dtype == torch.float32:
        out = torch.empty_like(t, memory_format=torch.contiguous_format)
        N.call("dq_add_mul", t.contiguous(), 1.0, 0.5, out, t.numel())
        return out
    return (t + 1) * 0.5


def identity(t, *args, **kwargs):
    return t


def extract(a, t, x_shape):
    b, *_ = t.shape
    out = a.gather(-1, t)
    return out.reshape(b, *((1,) * (len(x_shape) - 1)))


SAMPLERS = ("reference", "ddim", "dpm++2m")


def sampler_grid(T, N):
    """Time grid of the "ddim" / "dpm++2m" samplers: tau_i = rint((T-1) (1 - i/(N-1))^2), then raised so that the N
    points strictly decrease from T-1 to 0 (every integer when N = T).  The quadratic spacing keeps the log-SNR jumps
    at both ends of the cosine schedule small, where the reference's linear grid has its largest ones."""
    T, N = int(T), int(N)
    if not 2 <= N <= T:
        raise ValueError(f"the ODE samplers take 2 <= num_steps <= {T}, got {N}")
    tau = [int(np.rint((T - 1) * (1.0 - i / (N - 1)) ** 2)) for i in range(N)]
    for i in range(N - 2, -1, -1):
        tau[i] = max(tau[i], tau[i + 1] + 1)
    return tau


def ode_coefs(alpha_bars, taus, order):
    """Per-step arguments (alpha, sigma, c_x, c_d, w_cur, w_prev, last) of `dq_dpm_step` over the grid `taus`, in float64
    from the fp32 `alpha_bars` table.  Update i moves the state from tau_i to tau_{i+1} with h_i = lambda_{i+1} -
    lambda_i, lambda = log(alpha / sigma): c_x = sigma_{i+1} / sigma_i, c_d = -alpha_{i+1} expm1(-h_i).  The first and
    the final update (into tau = 0) are first order (w_cur = 1, w_prev = 0: DDIM with the true previous alpha_bar);
    order 2 is DPM-Solver++(2M) (arXiv:2211.01095, Algorithm 2) in between, r = h_{i-1} / h_i, w_cur = 1 + 1/(2r),
    w_prev = -1/(2r).  The last entry evaluates D at tau = 0 (`last` = 1)."""
    ab = np.asarray(alpha_bars, dtype=np.float32).astype(np.float64)[list(taus)]
    alpha, sigma = np.sqrt(ab), np.sqrt(1.0 - ab)
    lam = np.log(alpha / sigma)
    n = len(taus)
    steps = []
    for i in range(n - 1):
        h = lam[i + 1] - lam[i]
        w_cur, w_prev = 1.0, 0.0
        if order == 2 and 0 < i < n - 2:
            r = (lam[i] - lam[i - 1]) / h
            w_cur, w_prev = 1.0 + 0.5 / r, -0.5 / r
        steps.append((alpha[i], sigma[i], sigma[i + 1] / sigma[i], -alpha[i + 1] * math.expm1(-h), w_cur, w_prev, 0))
    steps.append((alpha[-1], sigma[-1], 0.0, 0.0, 1.0, 0.0, 1))
    return [tuple(float(v) for v in s[:6]) + (s[6],) for s in steps]


def _sic_loss(x0_like, ms1_n):
    """MS1 summary-ion-chromatogram loss over the RT profiles (sum / mean / max over mz, each divided by its global
    maximum, MSE against the normalised MS1 chromatogram): see oracle/dquartic_oracle.py:sic_loss for the definition."""
    tgt = ms1_n / torch.max(ms1_n)
    total = None
    for f in (lambda v: v.sum(-1), lambda v: v.mean(-1), lambda v: v.max(-1).values):
        sic = f(x0_like)
        term = torch.mean((sic / torch.max(sic) - tgt) ** 2)
        total = term if total is None else total + term
    return total


class _MSEFn(torch.autograd.Function):
    """mean((pred - target)^2) with the gradient produced in the same pass (F.mse_loss, model.py:361)."""

    @staticmethod
    def forward(ctx, pred, target):
        pred = pred.contiguous()
        target = target.contiguous()
        n = pred.numel()
        acc = torch.zeros(1, dtype=torch.float64, device=pred.device)
        d = torch.empty_like(pred)
        N.call("dq_mse", pred, target, acc, d, 2.0 / n, n)
        ctx.save_for_backward(d)
        return (acc / n).to(torch.float32).reshape(())

    @staticmethod
    def backward(ctx, g):
        (d,) = ctx.saved_tensors
        out = torch.empty_like(d)   # d * g in one kernel, the scalar stays on the device (no .item() sync)
        N.call("dq_scale_by", d, g.reshape(1).float().contiguous(), out, d.numel())
        return out, None


class DDIMDiffusionModel(ModelInterface):
    def __init__(
        self,
        model_class,
        num_timesteps=1000,
        beta_schedule_type="cosine",
        pred_type="eps",
        auto_normalize=True,
        ms1_loss_weight=0.0,
        device="cuda",
        **kwargs,
    ):
        super().__init__()
        self.model = None
        self.build(model_class, **kwargs)
        self.num_timesteps = num_timesteps
        self.device = device

        betas64 = get_linear_beta_schedule(num_timesteps) if beta_schedule_type == "linear" else get_cosine_beta_schedule(num_timesteps)
        self.betas = betas64.to(device).to(torch.float32)
        self.alphas = get_alphas(self.betas).to(torch.float32)
        # cumprod on the CPU in fp32, like the reference's CPU run, then moved: keeps the table bit-identical
        self.alpha_bars = get_alpha_bars(self.alphas.cpu()).to(torch.float32).to(device)
        self._ab_host = self.alpha_bars.detach().cpu().numpy().astype(np.float32)

        snr = self.alpha_bars / (1 - self.alpha_bars)
        if pred_type == "eps":
            self.loss_weight = torch.ones_like(snr)
        elif pred_type == "x0":
            self.loss_weight = snr
        else:
            raise ValueError(f"Unknown pred_type: {pred_type}")

        self.auto_normalize = auto_normalize
        self.normalize = normalize_to_neg_one_to_one if auto_normalize else identity
        self.unnormalize = unnormalize_to_zero_to_one if auto_normalize else identity
        self.pred_type = pred_type
        self.ms1_loss_weight = ms1_loss_weight

    # ------------------------------------------------------------------------------------------ forward process
    def q_sample(self, x_0, t, noise=None):
        """sqrt(ab[t]) * x_0 + sqrt(1 - ab[t]) * noise (model.py:225-242); x_0 is taken as given (already normalised)."""
        x_0 = x_0.float()   # the kernels compute in fp32 (a float64 tensor must not be reinterpreted)
        if noise is None:
            noise = torch.randn_like(x_0)
        noise = noise.float()
        b = x_0.shape[0]
        out = torch.empty_like(x_0, memory_format=torch.contiguous_format)
        N.call("dq_qsample", x_0.contiguous(), noise.contiguous(), t.to(torch.long).contiguous(), self.alpha_bars, out,
               b, x_0.numel() // b, 0)
        return out

    def _q_sample_fused(self, x_0_raw, t, noise):
        b = x_0_raw.shape[0]
        out = torch.empty_like(x_0_raw, memory_format=torch.contiguous_format)
        N.call("dq_qsample", x_0_raw.contiguous(), noise.contiguous(), t.contiguous(), self.alpha_bars, out, b,
               x_0_raw.numel() // b, 1 if self.auto_normalize else 0)
        return out

    # ------------------------------------------------------------------------------------------ reverse process
    def _step_coefs(self, t):
        ab = self._ab_host
        one = np.float32(1.0)
        sa = np.sqrt(ab[t])
        s1m = np.sqrt(one - ab[t])
        if t > 0:
            sap = np.sqrt(ab[t - 1])  # index t-1 regardless of the sampling stride (model.py:284)
            s1mp = np.sqrt(one - ab[t - 1])
        else:
            sap, s1mp = one, np.float32(0.0)
        return float(sa), float(s1m), float(sap), float(s1mp)

    def p_sample(self, x_t, t, init_cond=None, attn_cond=None):
        if self.pred_type not in ("eps", "x0"):
            raise ValueError(f"Unknown pred_type: {self.pred_type}")
        batch_size = x_t.size(0)
        t = int(t)
        x_t = x_t.float()
        t_tensor = torch.full((batch_size,), t, device=x_t.device, dtype=torch.long)
        sa, s1m, sap, s1mp = self._step_coefs(t)
        out = self.model(x_t, t_tensor, init_cond, attn_cond)
        if self.pred_type == "eps":
            eps_pred = out.contiguous()
            x_prev = torch.empty_like(eps_pred)
            N.call("dq_ddim_step", x_t.contiguous(), eps_pred, x_prev, sa, s1m, sap, s1mp, 1 if t == 0 else 0,
                   eps_pred.numel())
            return x_prev, eps_pred
        # pred_type == "x0" (model.py:275-289): one fused kernel, the reference's eager op order
        x0_pred = out.contiguous()
        x_prev = torch.empty_like(x0_pred)
        eps_pred = torch.empty_like(x0_pred)
        N.call("dq_ddim_step_x0", x_t.contiguous(), x0_pred, x_prev, eps_pred, sa, s1m, sap, s1mp, 1 if t == 0 else 0,
               x0_pred.numel())
        return x_prev, eps_pred

    def _ode_sample(self, x_t, ms2_cond, ms1_cond, num_steps, order):
        """The "ddim" (order 1) / "dpm++2m" (order 2) loop: one model call and one fused `dq_dpm_step` per grid point,
        every coefficient a host float fixed before the loop (so the loop captures into a CUDA graph).  Returns the
        data prediction at tau = 0 and, when there is no MS2 conditioning to derive the noise map from, its epsilon."""
        if self.pred_type not in ("eps", "x0"):
            raise ValueError(f"Unknown pred_type: {self.pred_type}")
        taus = sampler_grid(self.num_timesteps, num_steps)
        steps = ode_coefs(self._ab_host, taus, order)
        x = x_t.float().contiguous()
        b, n = x.size(0), x.numel()
        d_hist = torch.empty_like(x)
        eps = torch.empty_like(x) if ms2_cond is None else None
        for t, (alpha, sigma, c_x, c_d, w_cur, w_prev, last) in zip(taus, steps):
            t_tensor = torch.full((b,), t, device=x.device, dtype=torch.long)
            out = self.model(x, t_tensor, ms2_cond, ms1_cond).contiguous()
            x_next = torch.empty_like(x)
            N.call("dq_dpm_step", x, out, d_hist, x_next, eps if last else None, alpha, sigma,
                   1 if self.pred_type == "x0" else 0, c_x, c_d, w_cur, w_prev, last, n)
            x = x_next
        return x, eps

    def sample(self, x_t, ms2_cond=None, ms1_cond=None, num_steps=1000, sampler="reference"):
        """Reverse process from x_t at t = T-1.  `sampler`: "reference" is the reference's loop bit for bit (its step
        lands on alpha_bars[t-1] whatever the stride, so it only solves the ODE at num_steps = T); "ddim" and "dpm++2m"
        solve the probability-flow ODE on `sampler_grid(T, num_steps)` with first / second order updates (`ode_coefs`)."""
        if sampler not in SAMPLERS:
            raise ValueError(f"unknown sampler {sampler!r}: expected one of {', '.join(SAMPLERS)}")
        if sampler != "reference" and not 2 <= int(num_steps) <= self.num_timesteps:
            raise ValueError(f"sampler {sampler!r} takes 2 <= num_steps <= {self.num_timesteps}, got {num_steps}")
        ms2_cond = self.normalize(ms2_cond) if ms2_cond is not None else None
        ms1_cond = self.normalize(ms1_cond) if ms1_cond is not None else None
        pred_noise = None
        if sampler != "reference":
            x_t, pred_noise = self._ode_sample(x_t, ms2_cond, ms1_cond, int(num_steps), 2 if sampler == "dpm++2m" else 1)
        else:
            time_steps = torch.linspace(self.num_timesteps - 1, 0, num_steps, dtype=torch.long).tolist()
            for t in time_steps:  # the step list lives on the host: no per-step device sync (reference: t.item())
                x_t, pred_noise = self.p_sample(x_t, t, ms2_cond, ms1_cond)
        if ms2_cond is not None and self.auto_normalize and x_t.is_cuda:
            xo = torch.empty_like(x_t)
            pn = torch.empty_like(x_t)
            N.call("dq_sample_finalize", x_t.contiguous(), ms2_cond.contiguous(), xo, pn, x_t.numel())
            return xo, pn
        x_t, pred_noise = self.unnormalize(x_t), self.unnormalize(pred_noise)
        if ms2_cond is not None:
            pred_noise = self.unnormalize(ms2_cond) - x_t
        return x_t, pred_noise

    # ------------------------------------------------------------------------------------------ window-sharded sampling
    @staticmethod
    def window_seed(seed, window_id):
        """Seed of window `window_id`'s Philox stream: x_T depends on (seed, window id) only - not on the number of
        GPUs, the sharding or the chunking (SURVEY.md §8e)."""
        return (int(seed) * 0x9E3779B97F4A7C15 + int(window_id) * 0xD1B54A32D192ED03 + 0x2545F4914F6CDD1D) & 0x7FFFFFFFFFFFFFFF

    @staticmethod
    def shard_windows(n_windows, rank, world):
        """Contiguous block of window indices [lo, hi) of `rank` (blocks differ by at most one window)."""
        base, rem = divmod(int(n_windows), int(world))
        lo = rank * base + min(rank, rem)
        return lo, lo + base + (1 if rank < rem else 0)

    def sample_windows(self, window_ids, cond_fn, seed=0, num_steps=50, chunk=32, rank=None, world=None, out=None,
                       return_noise=False, cuda_graph=True, sampler="reference"):
        """DDIM-sample the DIA windows `window_ids` (model.py:293-324 per window; model_interface.py:1125-1150 returns
        item [0] only - here every window is kept).

        Sharding: with `rank` / `world` (default: torch.distributed's, else 0 / 1) this process samples the contiguous
        block `shard_windows(len(window_ids), rank, world)` of the list; there is NO collective, results stay on the host
        of each rank.  `cond_fn(ids) -> (ms2_cond (n, rt, mz), ms1_cond (n, rt))` supplies the conditioning of a chunk as
        tensors on `self.device` (values in [0, 1], as `sample` expects).  x_T of a window is drawn from a generator
        seeded with `window_seed(seed, id)`.  Windows stream through the sampler `chunk` at a time; the 50-step loop of a
        full chunk is captured ONCE in a CUDA graph (fixed shapes: the scalar coefficients and timesteps of every step
        are baked in) and replayed per chunk; results are copied to pinned host memory on a side stream while the next
        chunk runs.  `sampler` is passed to `sample`.  Returns (ids of this rank, maps (n_local, rt, mz) on the
        host[, pred_noise])."""
        dist = torch.distributed
        if rank is None or world is None:
            on = dist.is_available() and dist.is_initialized()
            rank, world = (dist.get_rank(), dist.get_world_size()) if on else (0, 1)
        ids_all = [int(w) for w in window_ids]
        lo, hi = self.shard_windows(len(ids_all), rank, world)
        ids = ids_all[lo:hi]
        dev = torch.device(self.device)
        self.model.eval()
        n = len(ids)
        if n == 0:
            e = out if out is not None else torch.empty(0)
            return (ids, e, torch.empty(0)) if return_noise else (ids, e)
        c2_0, c1_0 = cond_fn(ids[:1])
        rt, mz = c2_0.shape[1], c2_0.shape[2]
        if out is None:
            out = torch.empty((n, rt, mz), dtype=torch.float32).pin_memory()
        out_noise = torch.empty((n, rt, mz), dtype=torch.float32).pin_memory() if return_noise else None
        copy_stream = torch.cuda.Stream(device=dev)
        chunk = max(1, min(int(chunk), n))

        def draw_xT(chunk_ids, buf):
            for k, w in enumerate(chunk_ids):
                g = torch.Generator(device=dev)
                g.manual_seed(self.window_seed(seed, w))
                buf[k].normal_(generator=g)

        # static buffers of the captured graph
        xT = torch.empty((chunk, rt, mz), dtype=torch.float32, device=dev)
        c2 = torch.empty_like(xT)
        c1 = torch.empty((chunk, rt), dtype=torch.float32, device=dev)
        graph, res, stage = None, None, None
        pending = []
        with torch.no_grad():
            for s in range(0, n, chunk):
                cid = ids[s:s + chunk]
                nb = len(cid)
                a, b1 = cond_fn(cid)
                if nb == chunk:
                    draw_xT(cid, xT)
                    c2.copy_(a)
                    c1.copy_(b1)
                    if cuda_graph and graph is None and n >= 2 * chunk:
                        self.sample(xT.clone(), c2, c1, num_steps=min(2, num_steps), sampler=sampler)   # warm-up outside the capture
                        torch.cuda.synchronize(dev)
                        graph = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(graph):
                            res = self.sample(xT, c2, c1, num_steps=num_steps, sampler=sampler)
                    if graph is not None:
                        graph.replay()
                        x, pn = res
                    else:
                        x, pn = self.sample(xT, c2, c1, num_steps=num_steps, sampler=sampler)
                else:   # ragged last chunk: eager
                    xt = torch.empty((nb, rt, mz), dtype=torch.float32, device=dev)
                    draw_xT(cid, xt)
                    x, pn = self.sample(xt, a.float().contiguous(), b1.float().contiguous(), num_steps=num_steps,
                                        sampler=sampler)
                cur = torch.cuda.current_stream(dev)
                if graph is not None and nb == chunk:
                    # the graph's output buffers are overwritten by the next replay: move the results to staging buffers
                    # (a device-to-device copy, ~0.1 ms) so that the next replay does not wait for the host copy
                    if stage is None:
                        stage = (torch.empty_like(xT), torch.empty_like(xT) if return_noise else None)
                    if pending:
                        cur.wait_event(pending[-1])          # the previous host copy has read the staging buffers
                    stage[0].copy_(x)
                    if return_noise:
                        stage[1].copy_(pn)
                    x, pn = stage
                ev = torch.cuda.Event()
                ev.record(cur)
                with torch.cuda.stream(copy_stream):
                    copy_stream.wait_event(ev)
                    out[s:s + nb].copy_(x[:nb], non_blocking=True)
                    if return_noise:
                        out_noise[s:s + nb].copy_(pn[:nb], non_blocking=True)
                    done = torch.cuda.Event()
                    done.record(copy_stream)
                pending.append(done)
        for e in pending:
            e.synchronize()
        return (ids, out, out_noise) if return_noise else (ids, out)

    # ------------------------------------------------------------------------------------------ validation
    @torch.no_grad()
    def denoising_loss(self, x0, ms2_cond, ms1_cond, t, noise):
        """Per-sample MSE of the network's own training target at given timesteps `t` (b,) and standard-normal `noise`
        (b, rt, mz), no gradient: x_t = dq_qsample(x0, t, noise) (with the auto-normalise of `train_step`), one forward
        pass, target = noise ("eps") or normalize(x0) ("x0"), squared error summed by dq_map_scores.  Without the
        `loss_weight[t]` factor and without the MS1 SIC term of `train_step`.  Returns (b,) float64."""
        if self.pred_type not in ("eps", "x0"):
            raise ValueError(f"Unknown pred_type: {self.pred_type}")
        x0 = x0.float().contiguous()
        noise = noise.float().contiguous()
        t = t.to(x0.device).long().contiguous()
        ms2_n = self.normalize(ms2_cond) if ms2_cond is not None else None
        ms1_n = self.normalize(ms1_cond) if ms1_cond is not None else None
        x_t = self._q_sample_fused(x0, t, noise)
        pred = self.model(x_t, t, ms2_n, ms1_n)
        target = noise if self.pred_type == "eps" else self.normalize(x0)
        return self.map_scores(pred, target)[:, 0] / (x0[0].numel())

    # ------------------------------------------------------------------------------------------ training step
    def train_step(self, x_0, ms2_cond=None, ms1_cond=None, noise=None, ms1_loss_weight=0.0, t=None):
        """model.py:326-406.  `t` (optional, not in the reference) injects the timesteps for parity tests."""
        if self.pred_type not in ("eps", "x0"):
            raise ValueError(f"Unknown pred_type: {self.pred_type}")
        batch_size = x_0.size(0)
        dev = x_0.device
        if t is None:
            t = torch.randint(0, self.num_timesteps, (batch_size,), device=dev).long()
        else:
            t = t.to(dev).long()
        x_0 = x_0.float()
        noise = torch.randn_like(x_0) if noise is None else self.normalize(noise.float())
        ms2_n = self.normalize(ms2_cond) if ms2_cond is not None else None
        ms1_n = self.normalize(ms1_cond) if ms1_cond is not None else None
        x_t = self._q_sample_fused(x_0.float(), t, noise)
        pred = self.model(x_t, t, ms2_n, ms1_n)
        if self.pred_type == "eps":
            primary = _MSEFn.apply(pred, noise)
        else:
            primary = _MSEFn.apply(pred, self.normalize(x_0))
        loss = primary
        if ms1_loss_weight and ms1_loss_weight > 0.0:
            # Secondary mode (default weight 0.0, dquartic_train_config.json:18).  The reference's own code raises
            # TypeError here (torch.max(dim=-1) returns a tuple, model.py:366-368): the semantics are the ones defined
            # and documented in oracle/dquartic_oracle.py:sic_loss; small (b, RT) reductions, composed with autograd.
            x0_like = (x_t - pred) if self.pred_type == "eps" else pred
            loss = (1 - ms1_loss_weight) * primary + ms1_loss_weight * _sic_loss(x0_like, ms1_n)
        return loss * extract(self.loss_weight, t, (batch_size,))
