"""Drop-in for ``diffusion.SO3Diffusion`` / ``ProjectedSO3Diffusion`` of the reference
(diffusion.py:280-429): same constructor, method names, buffer names (state-dict compatible) and
shapes, with the manifold arithmetic of every step fused into one sm_100a kernel.

What changes underneath (SURVEY.md section 3):
  * the reference rebuilds a (1000, B) fp64 density table on every ``p_losses`` / ``q_sample`` call
    and a (1000, 1) one on every reverse step (distributions.py:11-31).  There are only T distinct
    eps values in a schedule, so two (T, 999) CDF tables (forward eps_t, posterior sigma_t) are built
    once per device by one kernel launch each and indexed by t inside the fused kernels;
  * ``p_losses``: ONE kernel draws the noise (device Philox), computes x_t = so3_scale(x0, a_t) @ noise
    and the regression target vee(log noise)/eps_t (known in closed form: angle * axis / eps);
  * ``p_sample``: ONE kernel does predict_start_from_noise, q_posterior, the posterior noise draw
    and the final composition (3 logs, 5 exps, 4 matmuls, 1 inverse-CDF lookup per particle);
    no host synchronisation (the reference's ``(t == 0).all()`` check is done per row on the device);
  * per-row t is honoured everywhere (the reference uses model_stdev[0] for the whole batch, Q7).
The denoiser stays a stock PyTorch module.
"""
from functools import partial

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops
from .distributions import IGSO3xR3, IsotropicGaussianSO3
from .util import AffineGrad, AffineT, compose, rmat_dist, se3_scale, so3_scale


def exists(x):
    return x is not None


def default(val, d):
    if exists(val):
        return val
    return d() if callable(d) else d


def extract(a, t, x_shape):
    """denoising_diffusion_pytorch.py:268-271."""
    b, *_ = t.shape
    out = a.gather(-1, t)
    return out.reshape(b, *((1,) * (len(x_shape) - 1)))


def cosine_beta_schedule(timesteps, s=0.008):
    """denoising_diffusion_pytorch.py:278-288 (https://openreview.net/forum?id=-NEXDKk8gZ)."""
    steps = timesteps + 1
    x = np.linspace(0, steps, steps)
    alphas_cumprod = np.cos(((x / steps) + s) / (1 + s) * np.pi * 0.5) ** 2
    alphas_cumprod = alphas_cumprod / alphas_cumprod[0]
    betas = 1 - (alphas_cumprod[1:] / alphas_cumprod[:-1])
    return np.clip(betas, a_min=0, a_max=0.999)


class SO3Diffusion(nn.Module):
    def __init__(self, denoise_fn, timesteps=1000, loss_type="skewvec", betas=None, reference_quirks=False):
        super().__init__()
        self.denoise_fn = denoise_fn
        self.reference_quirks = bool(reference_quirks)

        # ---- schedule buffers, diffusion.py:57-92 (numpy float64 -> float32 buffers) ------------
        if exists(betas):
            betas = betas.detach().cpu().numpy() if isinstance(betas, torch.Tensor) else betas
        else:
            betas = cosine_beta_schedule(timesteps)
        alphas = 1.0 - betas
        alphas_cumprod = np.cumprod(alphas, axis=0)
        alphas_cumprod_prev = np.append(1.0, alphas_cumprod[:-1])
        (timesteps,) = betas.shape
        self.num_timesteps = int(timesteps)
        self.loss_type = loss_type
        to_torch = partial(torch.tensor, dtype=torch.float32)
        self.register_buffer("betas", to_torch(betas))
        self.register_buffer("alphas_cumprod", to_torch(alphas_cumprod))
        self.register_buffer("alphas_cumprod_prev", to_torch(alphas_cumprod_prev))
        self.register_buffer("sqrt_alphas_cumprod", to_torch(np.sqrt(alphas_cumprod)))
        self.register_buffer("sqrt_one_minus_alphas_cumprod", to_torch(np.sqrt(1.0 - alphas_cumprod)))
        self.register_buffer("log_one_minus_alphas_cumprod", to_torch(np.log(1.0 - alphas_cumprod)))
        self.register_buffer("sqrt_recip_alphas_cumprod", to_torch(np.sqrt(1.0 / alphas_cumprod)))
        self.register_buffer("sqrt_recipm1_alphas_cumprod", to_torch(np.sqrt(1.0 / alphas_cumprod - 1)))
        posterior_variance = betas * (1.0 - alphas_cumprod_prev) / (1.0 - alphas_cumprod)
        self.register_buffer("posterior_variance", to_torch(posterior_variance))
        self.register_buffer("posterior_log_variance_clipped", to_torch(np.log(np.maximum(posterior_variance, 1e-20))))
        self.register_buffer("posterior_mean_coef1", to_torch(betas * np.sqrt(alphas_cumprod_prev) / (1.0 - alphas_cumprod)))
        self.register_buffer("posterior_mean_coef2", to_torch((1.0 - alphas_cumprod_prev) * np.sqrt(alphas) / (1.0 - alphas_cumprod)))
        self.register_buffer("identity", torch.eye(3))  # diffusion.py:283

        # global row index of this process's first batch row: makes the Philox draws of a sharded
        # batch independent of the number of GPUs (set by the multi-GPU harness)
        self.row_offset = 0
        self.fuse_denoiser = True  # p_sample runs a RotPredict denoiser inside the reverse-step kernel when it can
        self.fused_loop = True       # p_sample_loop(cuda_graph=True) with a fusable RotPredict: all T steps in ONE launch
        self._tables = {}  # schedule key -> (fwd_cdf, post_cdf, t_range)
        self._guides = {}  # schedule key -> (fwd_guide, post_guide)

    # ---- per-schedule CDF tables -----------------------------------------------------------------
    def tables(self):
        """(fwd_cdf (T,999) for eps_t = sqrt(1-abar_t),  post_cdf (T,999) for sigma_t,  arange(T))."""
        dev = self.betas.device
        key = self._schedule_key()
        if key not in self._tables:
            if dev.type != "cuda":
                raise RuntimeError("SO3Diffusion must be moved to a CUDA device (.to('cuda')); there is no CPU path")
            self._tables.clear()  # a stale schedule's tables (load_state_dict / in-place edits / .to()) are dropped, not kept
            self._guides.clear()
            fwd = ops.igso3_cdf_table(self.sqrt_one_minus_alphas_cumprod, self.reference_quirks)
            sigma = (0.5 * self.posterior_log_variance_clipped).exp()  # diffusion.py:324
            post = ops.igso3_cdf_table(sigma, self.reference_quirks)
            self._tables[key] = (fwd, post, torch.arange(self.num_timesteps, device=dev))
            self._guides[key] = (ops.igso3_cdf_guide(fwd), ops.igso3_cdf_guide(post))
        return self._tables[key]

    def _schedule_key(self):
        """Identity of the buffers the CDF tables are derived from: device, storage and in-place version counter.
        `load_state_dict` (copy_ into the buffers), in-place assignment and `.to(device)` all change it, so q_sample /
        p_sample can never draw noise from the tables of a schedule that is no longer the module's."""
        a, b = self.sqrt_one_minus_alphas_cumprod, self.posterior_log_variance_clipped
        return (str(a.device), a.data_ptr(), a._version, b.data_ptr(), b._version, bool(self.reference_quirks))

    def guides(self):
        """(fwd_guide, post_guide): the (T, 2051, 4) search records of the two CDF tables."""
        self.tables()
        return self._guides[self._schedule_key()]

    # ---- forward process ----------------------------------------------------------------------
    def q_mean_variance(self, x_start, t):
        """diffusion.py:285-289 (so3_lerp(I, x, w) == so3_scale(x, w))."""
        mean = so3_scale(x_start, self.sqrt_alphas_cumprod[t])
        variance = extract(1.0 - self.alphas_cumprod, t, x_start.shape)
        log_variance = extract(self.log_one_minus_alphas_cumprod, t, x_start.shape)
        return mean, variance, log_variance

    def q_sample(self, x_start, t, noise=None):
        """diffusion.py:339-346."""
        if noise is None:
            fwd, _, _ = self.tables()
            return ops.q_sample_fused(x_start, t, self.sqrt_alphas_cumprod, self.sqrt_one_minus_alphas_cumprod, fwd,
                                      row_offset=self.row_offset, want_target=False, guide=self.guides()[0])["x_t"]
        return ops.q_sample_given(x_start, t, self.sqrt_alphas_cumprod, noise)

    # ---- device-resident noise seed (CUDA-graph capturable training steps) --------------------------
    def use_device_seed(self, enable=True):
        """Keep the forward-noising seed in a device tensor that every `noise_and_target` call bumps by one ON THE
        DEVICE before its launch: the call sequence is then free of host-side RNG state, so a training step captured in
        a CUDA graph draws fresh noise on every replay (eager calls behave the same way).  Returns the seed tensor."""
        if not enable:
            self.__dict__.pop("_device_seed", None)
            return None
        dev = self.betas.device
        if dev.type != "cuda":
            raise RuntimeError("use_device_seed needs the process on a CUDA device")
        if self.__dict__.get("_device_seed") is None or self._device_seed.device != dev:
            seed, off = ops.rng.next()
            mixed = (seed + 0x9E3779B97F4A7C15 * (off + 1)) & 0x7FFFFFFFFFFFFFFF
            self._device_seed = torch.full((1,), mixed, dtype=torch.int64, device=dev)
        return self._device_seed

    def make_graphed_train_step(self, optimizer, example_x, warmup=3, sync_grads=None):
        """so3_train.py:70-76 / bingham_train.py:88-95 as ONE CUDA graph: `loss = self(x); loss.backward(); optimizer.step()`
        is captured once for batches shaped like `example_x` (a tensor, or an `AffineT` for the SE(3) classes; the optimizer
        must be constructed with capturable=True) and the returned `step(x) -> loss` copies x into the graph's input and
        replays it.  At the reference's batch sizes the eager step is launch-bound (~50 launches, 1.05 ms); the replay takes
        0.18 ms at batch 256 (tests/tools/probe_train.py).
        Noise comes from the device-resident seed (use_device_seed), step indices from torch's graph-safe generator.

        Data-parallel training (BASELINE cfg 4): with `sync_grads` (default: a process group with more than one rank is
        initialised) the gradients are flattened into ONE bucket, all-reduced over the ranks by a captured NCCL launch and
        averaged before the optimizer step -- what DistributedDataParallel does with its hooks, but inside the graph, so
        a replay is still one host call.  The denoiser must then be the bare module (not a DDP wrapper), initialised
        identically on every rank; every rank must use its own `row_offset`."""
        import torch.distributed as dist

        if sync_grads is None:
            sync_grads = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
        world = dist.get_world_size() if sync_grads else 1
        self.use_device_seed()
        static_x = example_x.detach().clone()
        dev = static_x.device
        params = [p for group in optimizer.param_groups for p in group["params"]]

        def one():
            optimizer.zero_grad(set_to_none=True)
            loss = self(static_x)
            loss.backward()
            if sync_grads:
                live = [p for p in params if p.grad is not None]
                flat = torch.cat([p.grad.reshape(-1) for p in live])
                dist.all_reduce(flat)                                   # captured: one bucket, one NCCL launch
                flat.mul_(1.0 / world)
                off = 0
                for p in live:
                    p.grad.copy_(flat[off:off + p.numel()].view_as(p.grad))
                    off += p.numel()
            optimizer.step()
            return loss

        with torch.cuda.device(dev):  # capture on the data's device even if it is not the process's current one
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                for _ in range(max(1, warmup)):
                    one()
            torch.cuda.current_stream(dev).wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            optimizer.zero_grad(set_to_none=True)
            with torch.cuda.graph(graph):
                static_loss = one()

        def step(x):
            static_x.copy_(x)
            graph.replay()
            return static_loss

        step.graph, step.static_x, step.sync_grads = graph, static_x, bool(sync_grads)
        return step

    def noise_and_target(self, x_start, t, want_noise=False, want_score=False):
        """One fused launch: noise ~ IGSO3(eps_t), x_t, and the 'skewvec' target vee(log noise)/eps_t
        (diffusion.py:349-355)."""
        fwd, _, _ = self.tables()
        dseed = self.__dict__.get("_device_seed")
        if dseed is not None and not (want_noise or want_score):
            dseed.add_(1)                                    # a captured kernel: every replay uses the next seed
            return ops.q_sample_fused(x_start, t, self.sqrt_alphas_cumprod, self.sqrt_one_minus_alphas_cumprod, fwd, seed=dseed, rng_offset=0,
                                      row_offset=self.row_offset, want_target=True, guide=self.guides()[0])
        return ops.q_sample_fused(x_start, t, self.sqrt_alphas_cumprod, self.sqrt_one_minus_alphas_cumprod, fwd,
                                  row_offset=self.row_offset, want_target=True, want_noise=want_noise, want_score=want_score,
                                  guide=self.guides()[0])

    # ---- reverse process ----------------------------------------------------------------------
    def predict_start_from_noise(self, x_t, t, noise):
        """diffusion.py:291-297."""
        _, x0_hat = ops.p_sample_fused(x_t, noise.detach(), t, self.sqrt_recip_alphas_cumprod, self.sqrt_recipm1_alphas_cumprod,
                                       self.posterior_mean_coef1, self.posterior_mean_coef2, post_cdf=None, want_x0_hat=True)
        return x0_hat

    def q_posterior(self, x_start, x_t, t):
        """diffusion.py:299-306."""
        c_1 = so3_scale(x_start, self.posterior_mean_coef1[t])
        c_2 = so3_scale(x_t, self.posterior_mean_coef2[t])
        posterior_mean = compose(c_1, c_2)
        posterior_variance = extract(self.posterior_variance, t, t.shape)
        posterior_log_variance_clipped = extract(self.posterior_log_variance_clipped, t, t.shape)
        return posterior_mean, posterior_variance, posterior_log_variance_clipped

    def _denoise(self, x, t):
        b = x.shape[0]
        t_full = t if t.numel() == b else t.expand(b)
        return self.denoise_fn(x, t_full)

    def _fused_denoiser(self, x, t):
        """(blob, c1_table) when `denoise_fn` is a RotPredict the fused kernel can run for this call, else None."""
        from .denoiser import RotPredict

        fn = self.denoise_fn
        if self.fuse_denoiser and type(self) in (SO3Diffusion,) and isinstance(fn, RotPredict) and t.numel() == 1 and fn.fusable():
            return fn.packed(self.num_timesteps)
        return None

    def p_mean_variance(self, x, t, clip_denoised: bool = False):
        """diffusion.py:308-313."""
        predict = self._denoise(x, t)
        model_mean = ops.p_sample_fused(x, predict, t, self.sqrt_recip_alphas_cumprod, self.sqrt_recipm1_alphas_cumprod,
                                        self.posterior_mean_coef1, self.posterior_mean_coef2, post_cdf=None)
        t_b = t if t.numel() == x.shape[0] else t.expand(x.shape[0])
        return model_mean, extract(self.posterior_variance, t_b, t_b.shape), extract(self.posterior_log_variance_clipped, t_b, t_b.shape)

    @torch.no_grad()
    def p_sample(self, x, t, clip_denoised=False, repeat_noise=False):
        """diffusion.py:315-326.  t: (B,) or (1,) int64.  One fused kernel after the denoiser; rows
        with t == 0 get no noise (checked on the device, no host sync)."""
        _, post, _ = self.tables()
        fused = self._fused_denoiser(x, t)
        if fused is not None:  # RotPredict + shared step: denoiser and reverse step in ONE tensor-core kernel
            blob, c1 = fused
            return ops.rotpredict_p_sample_fused(x, blob, c1, t, self.sqrt_recip_alphas_cumprod, self.sqrt_recipm1_alphas_cumprod,
                                                 self.posterior_mean_coef1, self.posterior_mean_coef2, post_cdf=post,
                                                 row_offset=self.row_offset)
        predict = self._denoise(x, t)
        return ops.p_sample_fused(x, predict, t, self.sqrt_recip_alphas_cumprod, self.sqrt_recipm1_alphas_cumprod,
                                  self.posterior_mean_coef1, self.posterior_mean_coef2, post_cdf=post, post_guide=self.guides()[1],
                                  row_offset=self.row_offset)

    # ---- the whole reverse process as ONE CUDA graph ---------------------------------------------
    def _p_sample_seeded(self, x, t, seed_buf, step):
        """p_sample with the Philox seed in device memory (`seed_buf`, int64[1]) and rng_offset = step: capturable,
        and a replay draws fresh noise once seed_buf has been rewritten."""
        _, post, _ = self.tables()
        fused = self._fused_denoiser(x, t)
        if fused is not None:
            blob, c1 = fused
            return ops.rotpredict_p_sample_fused(x, blob, c1, t, *self._sched4(), post_cdf=post, seed=seed_buf, rng_offset=step,
                                                 row_offset=self.row_offset)
        return ops.p_sample_fused(x, self._denoise(x, t), t, *self._sched4(), post_cdf=post, seed=seed_buf, rng_offset=step,
                                  row_offset=self.row_offset)

    def _sched4(self):
        return (self.sqrt_recip_alphas_cumprod, self.sqrt_recipm1_alphas_cumprod, self.posterior_mean_coef1, self.posterior_mean_coef2)

    def _seeded_steps(self, x, seed_buf, first=None):
        _, _, t_range = self.tables()
        steps = list(reversed(range(self.num_timesteps)))
        for i in steps if first is None else steps[:first]:
            x = self._p_sample_seeded(x, t_range[i:i + 1], seed_buf, i)
        return x

    def _p_sample_loop_graph(self, x):
        """Capture the T launches of the loop once per (batch shape, denoiser, weights) and replay them: the loop is
        launch-bound for the batch sizes the reference samples (bingham_test.py:25, 20 000 particles: ~10 us of GPU work
        per step), and a replay costs one launch.  Noise differs between replays because the kernels read the seed
        from `seed_buf` when they run (so3d_p_sample_dseed_f32 / so3d_rotpredict_p_sample_dseed_f32; the SE(3) classes
        supply their own step through `_p_sample_seeded`: so3d_se3_p_sample_dseed_f32)."""
        dev = x.device
        fn = self.denoise_fn
        probe = self._fused_denoiser(x, self.tables()[2][:1])          # (re)packs the weights if they changed
        if probe is not None and self.fused_loop:
            # RotPredict on the tensor-core route: no graph needed, the kernel itself runs all T steps in one launch
            seed, off = ops.rng.next()
            mixed = (seed + 0x9E3779B97F4A7C15 * (off + 1)) & 0xFFFFFFFFFFFFFFFF
            return ops.rotpredict_p_sample_loop(x, probe[0], probe[1], self.num_timesteps - 1, 0, *self._sched4(), self.tables()[1], mixed,
                                                row_offset=self.row_offset)
        packed_key = fn._packed[0] if probe is not None else None
        # everything the captured launches bake in: shapes, the denoiser object and its train/eval mode, the packed weights,
        # the projection closure of the Projected* classes (aircraft_test.py:73 sets a new one per item), the schedule
        key = (tuple(x.shape), str(dev), id(fn), bool(getattr(fn, "training", False)), packed_key, id(self.__dict__.get("projection")),
               self.row_offset, bool(self.fuse_denoiser), self.num_timesteps, self._schedule_key())
        cache = self.__dict__.setdefault("_loop_graphs", {})
        ent = cache.get(key)
        if ent is None:
            if len(cache) >= 4:
                cache.pop(next(iter(cache)))
            seed_buf = torch.zeros(1, dtype=torch.int64, device=dev)
            x_in = x.clone()
            with torch.cuda.device(dev):  # capture on the data's device even if it is not the process's current one
                side = torch.cuda.Stream(dev)
                side.wait_stream(torch.cuda.current_stream(dev))
                with torch.cuda.stream(side):                           # warm-up off the capture: lazy init, allocator
                    self._seeded_steps(x_in, seed_buf, first=3)
                torch.cuda.current_stream(dev).wait_stream(side)
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    x_out = self._seeded_steps(x_in, seed_buf)
            ent = (graph, x_in, seed_buf, x_out, probe, self.__dict__.get("projection"))  # keeps packed weights / the projection alive (ids stay unique)
            cache[key] = ent
        graph, x_in, seed_buf, x_out = ent[:4]
        seed, off = ops.rng.next()
        mixed = (seed + 0x9E3779B97F4A7C15 * (off + 1)) & 0xFFFFFFFFFFFFFFFF
        seed_buf.fill_(mixed - (1 << 64) if mixed >= (1 << 63) else mixed)
        x_in.copy_(x)
        graph.replay()
        return x_out.clone()

    @torch.no_grad()
    def p_sample_loop(self, shape, init="igso3_1", progress=False, cuda_graph=False):
        """diffusion.py:328-337.  init='igso3_1' is what the reference does (IGSO3(eps=1) samples,
        despite its comment); init='haar' starts from Haar-uniform rotations (SURVEY Q11).
        cuda_graph=True replays the whole loop as one captured CUDA graph (same distribution, its own noise stream)."""
        device = self.betas.device
        shape = tuple(shape)
        if init == "igso3_1":
            x = IsotropicGaussianSO3(torch.ones([], device=device)).sample(shape, row_offset=self.row_offset)
        elif init == "haar":
            x = ops.quat_to_rmat(torch.randn(*shape, 4, device=device))
        else:
            raise ValueError("init must be 'igso3_1' or 'haar'")
        if cuda_graph:
            return self._p_sample_loop_graph(x.contiguous())
        _, _, t_range = self.tables()
        steps = reversed(range(0, self.num_timesteps))
        if progress:
            from tqdm import tqdm

            steps = tqdm(steps, desc="sampling loop time step", total=self.num_timesteps)
        for i in steps:
            x = self.p_sample(x, t_range[i:i + 1])  # device-resident step index: no H2D copy per step
        return x

    @torch.no_grad()
    def reverse_process(self, x, pred=None, t_hi=None, t_lo=0):
        """The reverse chain x_{t_hi} -> x_{t_lo - 1} of `p_sample_loop` (diffusion.py:328-337) WITHOUT a denoiser in the loop:
        `pred` is None (zero prediction) or one fixed (...,3) prediction per particle.  With nothing but the manifold
        step between two steps, all of them run in ONE launch with the particles resident on chip
        (ops.p_sample_loop_fused); the result is bit-identical to p_sample_fused step by step.  This is the path
        BASELINE configs[2] times ("1000 steps x 2^24 particles", denoiser excluded); with a denoiser use p_sample_loop."""
        _, post, _ = self.tables()
        t_hi = self.num_timesteps - 1 if t_hi is None else int(t_hi)
        return ops.p_sample_loop_fused(x, pred, t_hi, int(t_lo), *self._sched4(), post, self.guides()[1], row_offset=self.row_offset)

    # ---- training loss ------------------------------------------------------------------------
    def p_losses(self, x_start, t, noise=None):
        """diffusion.py:348-369."""
        if noise is None:
            fused = self.noise_and_target(x_start, t)
            x_noisy, descaled_noise = fused["x_t"], fused["target"]
        else:
            eps = self.sqrt_one_minus_alphas_cumprod[t]
            x_noisy = self.q_sample(x_start, t, noise=noise)
            descaled_noise = ops.log_vec(noise) * (1 / eps)[..., None]
        x_recon = self.denoise_fn(x_noisy, t)
        if self.loss_type == "skewvec":
            loss = F.mse_loss(x_recon, descaled_noise)
        elif self.loss_type == "prevstep":
            posterior_mean, _, _ = self.q_posterior(x_start, x_noisy, t)
            step = compose(x_noisy, posterior_mean, trans_a=True)
            loss = rmat_dist(x_recon, step).pow(2.0).mean()
        else:
            raise RuntimeError(f"Unexpected loss_type: {self.loss_type}")  # the reference forgets to raise (Q9)
        return loss

    def forward(self, x, *args, **kwargs):
        b, *_, device = *x.shape, x.device
        t = torch.randint(0, self.num_timesteps, (b,), device=device).long()
        return self.p_losses(x, t, *args, **kwargs)


class ProjectedSO3Diffusion(SO3Diffusion):
    """diffusion.py:377-429: the denoiser sees projection(x) (e.g. a rotated point cloud)."""

    def __init__(self, denoise_fn, timesteps=1000, loss_type="skewvec", betas=None, reference_quirks=False):
        super().__init__(denoise_fn, timesteps=timesteps, loss_type=loss_type, betas=betas, reference_quirks=reference_quirks)
        self.register_buffer("identity", torch.eye(3))  # diffusion.py:380 (state-dict compatible)

    def _denoise(self, x, t):
        b = x.shape[0]
        t_full = t if t.numel() == b else t.expand(b)
        return self.denoise_fn(self.projection(x), t_full)

    @torch.no_grad()
    def p_sample_loop(self, shape, projection, init="haar", progress=False, cuda_graph=False):
        self.projection = projection
        return super().p_sample_loop(shape, init=init, progress=progress, cuda_graph=cuda_graph)

    def p_losses(self, x_start, t, noise=None):
        if noise is None:
            fused = self.noise_and_target(x_start, t)
            x_noisy, descaled_noise = fused["x_t"], fused["target"]
        else:
            eps = self.sqrt_one_minus_alphas_cumprod[t]
            x_noisy = self.q_sample(x_start, t, noise=noise)
            descaled_noise = ops.log_vec(noise) * (1 / eps)[..., None]
        if getattr(self, "check_finite", False):  # opt-in: the check is a host sync per step
            for name, val in (("x_noisy", x_noisy), ("descaled noise", descaled_noise)):
                if not torch.isfinite(val).all():
                    raise RuntimeError(f"{name} is not finite!")  # the reference builds these errors but never raises (Q9)
        x_recon = self.denoise_fn(self.projection(x_noisy), t)
        if self.loss_type not in ["backprop", "skewvec"]:
            raise RuntimeError(f"Unexpected loss_type: {self.loss_type}")
        return F.mse_loss(x_recon, descaled_noise)

    def forward(self, x, projection, *args, **kwargs):
        self.projection = projection
        return super().forward(x, *args, **kwargs)


class SE3Diffusion(SO3Diffusion):
    """diffusion.py:432-523: diffusion on SE(3) elements (`AffineT`): IGSO(3) noise on the rotation, Gaussian noise of
    scale eps * shift_scale on the translation, both halves of every step in ONE fused kernel
    (`so3d_se3_q_sample_f32` / `so3d_se3_p_sample_f32`).  Batches may carry extra frame dims, e.g. (B, N_res) protein
    backbone frames with a (B,) step index (prot_train.py): t broadcasts over the trailing batch dims.
    Same schedule buffers as the reference (it derives from GaussianDiffusion; state-dict compatible)."""

    def __init__(self, denoise_fn, timesteps=1000, loss_type="grad_mse", betas=None, shift_scale=75.0, reference_quirks=False):
        super().__init__(denoise_fn, timesteps=timesteps, loss_type=loss_type, betas=betas, reference_quirks=reference_quirks)
        self.shift_scale = shift_scale

    def _sigma(self):
        key = self._schedule_key()
        if getattr(self, "_sigma_cache", None) is None or self._sigma_cache[0] != key:
            self._sigma_cache = (key, (0.5 * self.posterior_log_variance_clipped).exp().contiguous())  # diffusion.py:481
        return self._sigma_cache[1]

    def _sched(self):
        return (self.sqrt_recip_alphas_cumprod, self.sqrt_recipm1_alphas_cumprod, self.posterior_mean_coef1, self.posterior_mean_coef2)

    # ---- forward process ----------------------------------------------------------------------
    def q_mean_variance(self, x_start, t):
        """diffusion.py:438-442."""
        mean = se3_scale(x_start, extract(self.sqrt_alphas_cumprod, t, t.shape))
        variance = extract(1.0 - self.alphas_cumprod, t, x_start.shape)
        log_variance = extract(self.log_one_minus_alphas_cumprod, t, x_start.shape)
        return mean, variance, log_variance

    def noise_and_target(self, x_start: AffineT, t):
        """One fused launch: noise ~ IGSO3xR3(eps_t, shift_scale), x_t, and both 'grad_mse' targets
        (diffusion.py:508-516).  -> (x_t: AffineT, target: AffineGrad)
        With `use_device_seed` the seed lives on the device and is bumped there before the launch (capturable)."""
        fwd, _, _ = self.tables()
        dseed = self.__dict__.get("_device_seed")
        if dseed is not None:
            dseed.add_(1)                                    # a captured kernel: every replay uses the next seed
        out = ops.se3_q_sample_fused(x_start.rot, x_start.shift, t, self.sqrt_alphas_cumprod, self.sqrt_one_minus_alphas_cumprod, fwd,
                                     self.shift_scale, seed=dseed, rng_offset=0 if dseed is not None else None, row_offset=self.row_offset,
                                     guide=self.guides()[0])
        return AffineT(out["rot"], out["shift"]), AffineGrad(out["target_rot"], out["target_shift"])

    def q_sample(self, x_start: AffineT, t, noise: AffineT = None):
        """diffusion.py:498-506."""
        if noise is None:
            return self.noise_and_target(x_start, t)[0]
        rot = ops.q_sample_given(x_start.rot, ops._rows_t(t, x_start.rot.shape[:-2], x_start.rot.device), self.sqrt_alphas_cumprod, noise.rot)
        scale = self.sqrt_alphas_cumprod[t].reshape(tuple(t.shape) + (1,) * (x_start.shift.dim() - t.dim()))
        return AffineT(rot, x_start.shift * scale + noise.shift)

    # ---- reverse process ----------------------------------------------------------------------
    def _step(self, x: AffineT, predict: AffineGrad, t, noise: bool):
        _, post, _ = self.tables()
        rot, shift = ops.se3_p_sample_fused(x.rot, x.shift, predict.rot_g, predict.shift_g, t, *self._sched(), self._sigma(), self.shift_scale,
                                            post_cdf=post if noise else None, post_guide=self.guides()[1] if noise else None,
                                            row_offset=self.row_offset)
        return AffineT(rot, shift)

    def predict_start_from_noise(self, x_t: AffineT, t, noise: AffineGrad):
        """diffusion.py:444-455."""
        rot = SO3Diffusion.predict_start_from_noise(self, x_t.rot, t, noise.rot_g)
        tb = t.reshape(tuple(t.shape) + (1,) * (x_t.shift.dim() - t.dim()))
        return AffineT(rot, x_t.shift * self.sqrt_recip_alphas_cumprod[tb] - noise.shift_g * self.sqrt_recipm1_alphas_cumprod[tb])

    def q_posterior(self, x_start: AffineT, x_t: AffineT, t):
        """diffusion.py:457-464."""
        c_1 = se3_scale(x_start, self.posterior_mean_coef1[t])
        c_2 = se3_scale(x_t, self.posterior_mean_coef2[t])
        posterior_mean = AffineT(compose(c_1.rot, c_2.rot), c_1.shift + c_2.shift)
        return posterior_mean, extract(self.posterior_variance, t, t.shape), extract(self.posterior_log_variance_clipped, t, t.shape)

    def _denoise(self, x: AffineT, t):
        return self.denoise_fn(x, t)

    def p_mean_variance(self, x: AffineT, t, clip_denoised: bool = False):
        """diffusion.py:466-471 (posterior mean of both halves in one launch)."""
        predict = self._denoise(x, t)
        mean = self._step(x, predict, t, noise=False)
        return mean, extract(self.posterior_variance, t, t.shape), extract(self.posterior_log_variance_clipped, t, t.shape)

    @torch.no_grad()
    def p_sample(self, x: AffineT, t, clip_denoised=False, repeat_noise=False):
        """diffusion.py:473-485: one fused kernel after the denoiser; rows with t == 0 get no noise (device-side check)."""
        return self._step(x, self._denoise(x, t), t, noise=True)

    def _p_sample_seeded(self, x: AffineT, t, seed_buf, step):
        """The step of the captured loop (SO3Diffusion._p_sample_loop_graph): the denoiser sees a (B,) step index as in the
        eager loop, the kernel the shared step `t` with the seed read from `seed_buf` and rng_offset = step."""
        _, post, _ = self.tables()
        predict = self._denoise(x, torch.full(x.rot.shape[:1], step, device=x.device, dtype=torch.long))
        rot, shift = ops.se3_p_sample_fused(x.rot, x.shift, predict.rot_g, predict.shift_g, t, *self._sched(), self._sigma(), self.shift_scale,
                                            post_cdf=post, seed=seed_buf, rng_offset=step, row_offset=self.row_offset)
        return AffineT(rot, shift)

    @torch.no_grad()
    def p_sample_loop(self, shape, init="haar", progress=False, cuda_graph=False):
        """diffusion.py:487-496 (the reference starts from rotations only; here the translation starts at
        N(0, shift_scale^2 I), the forward process's terminal law, like ProjectedSE3Diffusion does with N(0, I)).
        cuda_graph=True replays the whole loop as one captured CUDA graph (same distribution, its own noise stream)."""
        device = self.betas.device
        shape = tuple(shape)
        x = AffineT(self._init_rot(shape, init), torch.randn(*shape, 3, device=device) * self.shift_scale)
        return self._run_loop(x, shape, progress, cuda_graph)

    def _run_loop(self, x: AffineT, shape, progress, cuda_graph):
        if cuda_graph:
            return self._p_sample_loop_graph(AffineT(x.rot.contiguous(), x.shift.contiguous()))
        for i in self._steps(progress):
            x = self.p_sample(x, torch.full(shape[:1], i, device=x.device, dtype=torch.long))
        return x

    def _init_rot(self, shape, init):
        device = self.betas.device
        if init == "haar":
            return ops.quat_to_rmat(torch.randn(*shape, 4, device=device))
        if init == "igso3_1":
            return IsotropicGaussianSO3(torch.ones([], device=device)).sample(shape, row_offset=self.row_offset)
        raise ValueError("init must be 'igso3_1' or 'haar'")

    def _steps(self, progress):
        steps = reversed(range(0, self.num_timesteps))
        if progress:
            from tqdm import tqdm

            steps = tqdm(steps, desc="sampling loop time step", total=self.num_timesteps)
        return steps

    # ---- training loss ------------------------------------------------------------------------
    def p_losses(self, x_start: AffineT, t, noise=None):
        """diffusion.py:508-520."""
        x_noisy, target = self.noise_and_target(x_start, t)
        x_recon = self._denoise(x_noisy, t)
        if self.loss_type != "grad_mse":
            raise RuntimeError(f"Unexpected loss_type: {self.loss_type}")  # the reference forgets to raise (Q9)
        rot_g = x_recon.rot_g if hasattr(x_recon, "rot_g") else x_recon.rot
        shift_g = x_recon.shift_g if hasattr(x_recon, "shift_g") else x_recon.shift
        return F.mse_loss(shift_g, target.shift_g) + F.mse_loss(rot_g, target.rot_g)

    def forward(self, x: AffineT, *args, **kwargs):
        b, device = len(x), x.device
        t = torch.randint(0, self.num_timesteps, (b,), device=device).long()
        return self.p_losses(x, t, *args, **kwargs)


class ProjectedSE3Diffusion(SE3Diffusion):
    """diffusion.py:526-573: the denoiser sees projection(x)."""

    def __init__(self, denoise_fn, timesteps=1000, loss_type="grad_mse", betas=None, shift_scale=75.0, reference_quirks=False):
        super().__init__(denoise_fn, timesteps=timesteps, loss_type=loss_type, betas=betas, shift_scale=shift_scale, reference_quirks=reference_quirks)
        self.register_buffer("identity", torch.eye(3))  # diffusion.py:529 (state-dict compatible)

    def _denoise(self, x: AffineT, t):
        return self.denoise_fn(self.projection(x), t)

    @torch.no_grad()
    def p_sample_loop(self, shape, projection, init="haar", progress=False, cuda_graph=False):
        """diffusion.py:541-552: translation starts from N(0, I) as in the reference.  cuda_graph as in SE3Diffusion."""
        self.projection = projection
        device = self.betas.device
        shape = tuple(shape)
        x = AffineT(self._init_rot(shape, init), torch.randn(*shape, 3, device=device))
        return self._run_loop(x, shape, progress, cuda_graph)

    def forward(self, x: AffineT, projection, *args, **kwargs):
        self.projection = projection
        return super().forward(x, *args, **kwargs)


__all__ = ["SO3Diffusion", "ProjectedSO3Diffusion", "SE3Diffusion", "ProjectedSE3Diffusion", "extract", "cosine_beta_schedule",
           "exists", "default"]
