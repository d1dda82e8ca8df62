"""Drop-in for ``distributions.IsotropicGaussianSO3`` of the reference (distributions.py:8-81).

Same constructor / ``sample`` / ``log_prob`` / ``_eps_ft`` / ``mean`` / ``trap`` / ``trap_loc``
surface, CUDA float32 only, every method one fused sm_100a kernel:

  * the (999, *E) CDF table of distributions.py:15-30 is built on the device by one kernel
    (fp64 density -> fp32 trapezoid CDF, same dtype at every step as the reference) and only when
    something needs it (``sample`` / ``trap``), not in the constructor;
  * ``sample`` draws axis + uniform with a counter-based Philox stream on the device (the reference
    draws the axes with the CPU generator and copies them over, distributions.py:35), finds the
    angle by binary search (shared-memory CDF row for scalar eps) and applies Rodrigues' formula;
  * ``log_prob`` fuses axis-angle extraction, density and (saved for backward) d log f / d omega;
    per-row eps is supported (the reference raises, SURVEY Q2);
  * ``score`` is new: (d/d omega log f) * axis, the quantity the reference only reaches through
    autograd (distributions.py:186-190).

``mode`` selects the density evaluator: "closed" (the reference's 3-image closed form in its stable
rewrite), "series" (every row runs the L-term truncated series; rows where that alternating sum is
ill-conditioned in fp32 -- omega > 4.2 eps, cond > 14 -- are then replaced by the closed form, so the
result is <= 1e-5 relative on the whole E-set), "series_pure" (the raw fp32 series everywhere: error
~4 u cond, 6e-5 at omega = 5.66 eps), "auto" (default: closed form up to eps = 1, series above;
<= 1e-5 relative everywhere), "series_adaptive" (= "series", skipping zero-weight terms).
``reference_quirks=True`` builds the CDF table from the reference's literal overflowing expression
(density zeroed beyond omega > 709 eps^2/pi, SURVEY D5) so that samples match the reference at
tiny eps too.  Quirk Q1 (column-0 gather with batched eps) is a plain bug and is not reproduced.
``sampler`` selects how ``sample`` finds the angle: "table" (default: the reference's piecewise-linear inversion of the
999-point trapezoid CDF above, built per distinct eps) or "exact" (the inverse CDF of the IGSO(3) angle law itself, found
per row in registers with no table: |F(angle) - u| ~ 3e-7, and per-row eps costs 4 bytes per row instead of a 3996-byte
table row; ``trap`` / ``table`` still build the table if read).  The quirks belong to the table, so ``sampler="exact"``
with ``reference_quirks=True`` raises.
``rsample`` is the reparameterised draw: always the exact inverse CDF (whatever ``sampler`` says), differentiable w.r.t. eps
and the mean through one backward kernel.  At fixed (u, axis) the angle's derivative is dw/deps = -2 eps d log f / dw (the
heat equation turns the implicit derivative -(dF/deps)/p into the angle score), evaluated at the sampled angle.
``entropy`` is the entropy of the law w.r.t. normalised Haar measure (like ``rsample``, independent of the mean, ``mode``,
``series_terms`` and ``sampler``), differentiable w.r.t. eps: the kernel also writes dH/deps = 2 eps E[(d log f / dw)^2]
(de Bruijn's identity, the same heat equation), so the backward is one multiply.
"""
import torch
from torch.autograd.function import once_differentiable
from torch.distributions import Distribution, MultivariateNormal, Normal, constraints

from . import ops
from .util import AffineT


class _LogProb(torch.autograd.Function):
    @staticmethod
    def forward(ctx, rotations, eps, mode, L):
        logp, _, dlogf = ops.igso3_logp_score(rotations, eps, mode=mode, L=L, want_score=False, want_dlogf=True)
        ctx.save_for_backward(rotations, dlogf)
        return logp

    @staticmethod
    def backward(ctx, grad):
        rotations, dlogf = ctx.saved_tensors
        return ops.igso3_logp_bwd(rotations, dlogf, grad.contiguous()), None, None, None


class _RSample(torch.autograd.Function):
    """R = mean exp(w hat(a)), w = F^{-1}(u; eps) by the exact sampler; u and a are constants of the draw."""

    @staticmethod
    def forward(ctx, eps, mean, eps_rows, shape, u, axes, row_offset):
        seed, rng_offset = ops.rng.next()
        R, angle, axis = ops.igso3_sample_exact(eps_rows, shape, u=u, axes=axes, seed=seed, rng_offset=rng_offset,
                                                row_offset=row_offset, mean=mean, want_angle=True, want_axis=True)
        ctx.save_for_backward(eps_rows, mean, angle, axis, u)
        ctx.draw = (seed, rng_offset, row_offset)
        ctx.shapes = (eps.shape, None if mean is None else mean.shape)
        return R

    @staticmethod
    @once_differentiable
    def backward(ctx, grad):
        eps_rows, mean, angle, axis, u = ctx.saved_tensors
        seed, rng_offset, row_offset = ctx.draw
        eps_shape, mean_shape = ctx.shapes
        want_mean = mean is not None and ctx.needs_input_grad[1]
        g_eps, g_mean = ops.igso3_rsample_bwd(eps_rows, angle, axis, grad, u=u, seed=seed, rng_offset=rng_offset,
                                              row_offset=row_offset, mean=mean, want_mean_grad=want_mean)
        g_eps = g_eps.sum().reshape(eps_shape) if eps_rows.numel() == 1 else g_eps.sum_to_size(eps_shape)
        if want_mean:
            g_mean = g_mean.reshape(-1, 9).sum(0).reshape(mean_shape) if mean.numel() == 9 else g_mean.sum_to_size(mean_shape)
        return g_eps, g_mean, None, None, None, None, None


class _Entropy(torch.autograd.Function):
    """H(eps), with dH/deps from the same launch saved for the backward."""

    @staticmethod
    def forward(ctx, eps):
        H, dH = ops.igso3_entropy(eps, want_grad=ctx.needs_input_grad[0])
        ctx.save_for_backward(dH)
        return H

    @staticmethod
    @once_differentiable
    def backward(ctx, grad):
        (dH,) = ctx.saved_tensors
        return grad * dH


class IsotropicGaussianSO3(Distribution):
    arg_constraints = {"eps": constraints.positive}
    has_rsample = True

    def __init__(self, eps: torch.Tensor, mean: torch.Tensor = None, mode: str = "auto", series_terms: int = 2000,
                 reference_quirks: bool = False, sampler: str = "table"):
        if sampler not in ("table", "exact"):
            raise ValueError(f"sampler must be 'table' or 'exact' (got {sampler!r})")
        if sampler == "exact" and reference_quirks:
            raise ValueError("sampler='exact' draws from the IGSO(3) law itself; reference_quirks only shape the CDF table of "
                             "sampler='table'")
        if not isinstance(eps, torch.Tensor):
            raise TypeError("eps must be a torch.Tensor on a CUDA device")
        if not eps.is_cuda:
            raise RuntimeError("IsotropicGaussianSO3: eps must live on a CUDA device; this package has no CPU path")
        self.eps = eps.float() if eps.dtype != torch.float32 else eps
        self._mean = None if mean is None else mean.to(self.eps)
        self.eval_mode = mode
        self.series_terms = int(series_terms)
        self.reference_quirks = bool(reference_quirks)
        self.sampler = sampler
        self._table = None  # (E_flat, 999), built on first use
        super().__init__(batch_shape=self.eps.shape, validate_args=False)

    # -- CDF table (distributions.py:15-30) ------------------------------------------------------
    @property
    def table(self) -> torch.Tensor:
        """(numel(eps), 999): one contiguous CDF row per eps (transpose of the reference layout)."""
        if self._table is None:
            self._table = ops.igso3_cdf_table(self.eps.reshape(-1), self.reference_quirks)
        return self._table

    @property
    def trap(self) -> torch.Tensor:
        """Reference layout: (999, *E), or (999, 1) for scalar eps."""
        t = self.table.t()
        return t.reshape(ops.CDF_POINTS, *self.eps.shape) if self.eps.dim() > 0 else t

    @property
    def trap_loc(self) -> torch.Tensor:
        return ops.cdf_grid(self.eps.device)[2][:, None]

    @property
    def mean(self):
        if self._mean is None:
            return torch.eye(3, dtype=torch.float32, device=self.eps.device)
        return self._mean

    # -- sampling (distributions.py:33-51) -------------------------------------------------------
    @torch.no_grad()
    def sample(self, sample_shape=torch.Size(), *, u=None, axes=None, row_offset=0, return_angle=False):
        """Rotations of shape (*sample_shape, *eps.shape, 3, 3).
        u / axes: optional explicit uniforms / (un-normalised) axes, for reproducing given draws."""
        sample_shape = tuple(sample_shape)
        shape = sample_shape + tuple(self.eps.shape)
        if self._mean is not None and self._mean.dim() > 2:
            # a batched mean broadcasts against the noise like the reference's `self._mean @ rotations`
            # (distributions.py:50; e.g. IGSO3xR3(eps=sigma[0], mean=model_mean).sample() at diffusion.py:482 -> (B,3,3))
            shape = tuple(torch.broadcast_shapes(shape, self._mean.shape[:-2]))
        if self.sampler == "exact":
            eps = self.eps if self.eps.numel() == 1 else self.eps.expand(shape)
            return ops.igso3_sample_exact(eps, shape, u=u, axes=axes, row_offset=row_offset, mean=self._mean, want_angle=return_angle)
        if self.eps.dim() == 0:
            row_idx, row = None, 0
        else:
            row_idx = torch.arange(self.eps.numel(), device=self.eps.device).reshape(self.eps.shape).expand(shape)
            row = 0
        return ops.igso3_sample(self.table, shape, row_idx=row_idx, row=row, u=u, axes=axes, row_offset=row_offset,
                                mean=self._mean, want_angle=return_angle)

    def rsample(self, sample_shape=torch.Size(), *, u=None, axes=None, row_offset=0):
        """Reparameterised draw: rotations of shape (*sample_shape, *eps.shape, 3, 3) (broadcast against a batched mean, as in
        ``sample``), differentiable w.r.t. eps and the mean.  The angle always comes from the exact inverse CDF of the IGSO(3)
        law (with ``sampler="exact"`` the values are ``sample``'s, bit for bit, at the same seed).  u / axes are constants of
        the draw (no gradient flows to them).  The gradient w.r.t. eps is sign(eps) dw/d|eps|; at eps = 0 it is the eps -> 0+
        limit 2 x0(u), x0 the Maxwell quantile.  Once differentiable."""
        if self.reference_quirks:
            raise ValueError("rsample draws from the IGSO(3) law itself through the exact inverse CDF; reference_quirks only shape "
                             "the CDF table of sampler='table'")
        shape = tuple(sample_shape) + tuple(self.eps.shape)
        if self._mean is not None and self._mean.dim() > 2:
            shape = tuple(torch.broadcast_shapes(shape, self._mean.shape[:-2]))
        eps_rows = self.eps.detach()
        if eps_rows.numel() != 1:
            eps_rows = eps_rows.expand(shape)
        u = None if u is None else u.detach()
        axes = None if axes is None else axes.detach()
        return _RSample.apply(self.eps, self._mean, eps_rows, shape, u, axes, row_offset)

    def entropy(self):
        """Entropy of IGSO(3)(eps) w.r.t. normalised Haar measure, shape eps.shape, differentiable w.r.t. eps (so KL(q || Haar)
        = -entropy()).  The law's own entropy: independent of the mean, ``mode``, ``series_terms`` and ``sampler``.  Even in
        eps; eps = 0 gives -inf with gradient +inf (the 0+ limit 3/eps).  Once differentiable."""
        if self.reference_quirks:
            raise ValueError("entropy is that of the IGSO(3) law itself; reference_quirks only shape the CDF table of "
                             "sampler='table'")
        return _Entropy.apply(self.eps)

    # -- density (distributions.py:53-72) --------------------------------------------------------
    def _eps_ft(self, t: torch.Tensor) -> torch.Tensor:
        t = t.to(device=self.eps.device, dtype=torch.float32)
        if self.eps.numel() == 1:
            return ops.igso3_density(t.contiguous(), self.eps, mode=self.eval_mode, L=self.series_terms)
        shape = torch.broadcast_shapes(t.shape, self.eps.shape)
        return ops.igso3_density(t.expand(shape).contiguous(), self.eps.expand(shape).contiguous(), mode=self.eval_mode, L=self.series_terms)

    def log_prob(self, rotations):
        """distributions.py:74-77: log f_eps(angle(R)), shape (..., 1).  Differentiable w.r.t. rotations, not w.r.t. eps:
        with grad mode on and an eps that requires grad this raises instead of returning a result without that gradient."""
        if torch.is_grad_enabled() and isinstance(self.eps, torch.Tensor) and self.eps.requires_grad:
            raise NotImplementedError("IsotropicGaussianSO3.log_prob: the gradient w.r.t. eps is not implemented; pass eps.detach() "
                                      "or evaluate under torch.no_grad()")
        if torch.is_grad_enabled() and rotations.requires_grad:
            return _LogProb.apply(rotations, self.eps, self.eval_mode, self.series_terms)[..., None]
        logp, _, _ = ops.igso3_logp_score(rotations, self.eps, mode=self.eval_mode, L=self.series_terms, want_score=False)
        return logp[..., None]

    @torch.no_grad()
    def score(self, rotations):
        """(d log f / d omega) * axis, shape (..., 3): the Riemannian score in the body frame."""
        _, score, _ = ops.igso3_logp_score(rotations, self.eps, mode=self.eval_mode, L=self.series_terms, want_score=True)
        return score

    @torch.no_grad()
    def log_prob_and_score_host(self, rotations, out_logp=None, out_score=None, chunk_rows=1 << 20, pipeline=None):
        """Host-buffer entry point: `rotations` (n,3,3) is a (preferably pinned) HOST float32 tensor; returns HOST
        tensors logp (n,1) and score (n,3).  H2D copy, kernel and D2H copy are overlapped chunk by chunk
        (ops.HostScorePipeline).  If this distribution has per-row eps, a HOST copy of eps is streamed alongside."""
        n = rotations.shape[0]
        if rotations.is_cuda:
            raise ValueError("log_prob_and_score_host takes HOST tensors; use log_prob_and_score for device tensors")
        per_row = self.eps.numel() == n and n > 1
        if pipeline is None:
            pipeline = ops.HostScorePipeline(self.eps.device, chunk_rows=chunk_rows, per_row_eps=per_row)
        if out_logp is None:
            out_logp = torch.empty(n, dtype=torch.float32, pin_memory=True)
        if out_score is None:
            out_score = torch.empty(n, 3, dtype=torch.float32, pin_memory=True)
        heps = self._host_eps if per_row and getattr(self, "_host_eps", None) is not None else (self.eps.cpu() if per_row else self.eps)
        pipeline.run(rotations.contiguous(), heps, out_logp.reshape(n), out_score, mode=self.eval_mode, L=self.series_terms)
        return out_logp.reshape(n, 1), out_score

    @torch.no_grad()
    def log_prob_and_score(self, rotations):
        logp, score, _ = ops.igso3_logp_score(rotations, self.eps, mode=self.eval_mode, L=self.series_terms, want_score=True)
        return logp[..., None], score


class IGSO3xR3(Distribution):
    """distributions.py:84-110: product of IGSO3(eps) on the rotation and N(shift, (eps * shift_scale)^2 I) on the
    translation of an SE(3) element (`AffineT`).  `sample` draws both halves on the device; `rsample` too, differentiably.
    `entropy` adds the two halves' entropies."""

    arg_constraints = {"eps": constraints.positive}
    has_rsample = True

    def __init__(self, eps: torch.Tensor, mean: AffineT = None, shift_scale=1.0, mode: str = "auto"):
        self.eps = eps
        if mean is None:
            rot = torch.eye(3, device=eps.device).unsqueeze(0)
            shift = torch.zeros(*eps.shape, 3).to(eps)
            mean = AffineT(shift=shift, rot=rot)
        self._mean = mean.to(eps.device)
        self.shift_scale = shift_scale
        self.igso3 = IsotropicGaussianSO3(eps=eps, mean=self._mean.rot, mode=mode)
        self.r3 = Normal(loc=self._mean.shift, scale=eps[..., None] * shift_scale)
        super().__init__(validate_args=False)

    @torch.no_grad()
    def sample(self, sample_shape=torch.Size()):
        rot = self.igso3.sample(sample_shape)
        shift = self.r3.sample(sample_shape)
        return AffineT(rot, shift)

    def rsample(self, sample_shape=torch.Size()):
        """Reparameterised draw, differentiable w.r.t. eps and the mean: the rotation from ``IsotropicGaussianSO3.rsample``
        (exact inverse CDF), the shift from ``Normal.rsample``."""
        rot = self.igso3.rsample(sample_shape)
        shift = self.r3.rsample(sample_shape)
        return AffineT(rot, shift)

    def entropy(self):
        """Entropy of the product law: the IGSO(3) entropy plus that of the isotropic Gaussian shift, differentiable w.r.t. eps."""
        return self.igso3.entropy() + self.r3.entropy().sum(-1)

    def log_prob(self, value):
        rot_prob = self.igso3.log_prob(value.rot)      # (..., 1)
        shift_prob = self.r3.log_prob(value.shift)     # (..., 3)
        return rot_prob + shift_prob

    @property
    def mean(self):
        return self._mean


class Bingham(MultivariateNormal):
    """distributions.py:113-127: zero-mean Gaussian in R^4 pushed onto the unit quaternions (real part first).

    Same constructor as the reference (a MultivariateNormal whose `loc` is replaced by zeros).  On a CUDA device
    with a single (4,4) covariance, `rsample` / `sample` are ONE fused kernel (device Philox normals, L z,
    normalisation), and `sample_rmat` additionally fuses the `quat_to_rmat` the reference applies to every batch
    (bingham_train.py:88-90).  `z=` reproduces given standard-normal draws (parity tests).  Gradients w.r.t. the
    covariance take the stock torch route."""

    arg_constraints = {"covariance_matrix": constraints.positive_definite, "precision_matrix": constraints.positive_definite,
                       "scale_tril": constraints.lower_cholesky}
    support = constraints.real_vector

    def __init__(self, loc, covariance_matrix=None, precision_matrix=None, scale_tril=None, validate_args=None):
        loc = torch.zeros_like(loc)  # distributions.py:120: always zero-mean (antipodally symmetric)
        super().__init__(loc, covariance_matrix, precision_matrix, scale_tril, validate_args)
        self.row_offset = 0

    def _fused(self):
        st = self._unbroadcasted_scale_tril
        return st.is_cuda and st.dtype == torch.float32 and st.shape == (4, 4) and not (torch.is_grad_enabled() and st.requires_grad)

    def _require_cuda(self):
        if not self._unbroadcasted_scale_tril.is_cuda:
            raise RuntimeError("Bingham: the covariance must live on a CUDA device; this package has no CPU path "
                               "(the reference pins bingham_train.py to the CPU generator, bingham_train.py:52)")

    def rsample(self, sample_shape=torch.Size(), *, z=None):
        self._require_cuda()
        if self._fused():
            shape = tuple(sample_shape) + tuple(self.batch_shape)
            return ops.bingham_sample(self._unbroadcasted_scale_tril, shape, z=z, row_offset=self.row_offset)
        # batched covariances / gradients w.r.t. the covariance (reparameterised sample): torch ops ON THE DEVICE
        vals = super().rsample(sample_shape)
        return vals / vals.norm(dim=-1, keepdim=True)

    @torch.no_grad()
    def sample_rmat(self, sample_shape=torch.Size(), *, z=None):
        """quat_to_rmat(self.sample(sample_shape)) in one launch: (*sample_shape, 3, 3)."""
        self._require_cuda()
        if not self._fused():
            from .util import quat_to_rmat

            return quat_to_rmat(self.rsample(sample_shape))
        shape = tuple(sample_shape) + tuple(self.batch_shape)
        return ops.bingham_sample(self._unbroadcasted_scale_tril, shape, z=z, row_offset=self.row_offset, want_quat=False, want_rmat=True)


__all__ = ["IsotropicGaussianSO3", "IGSO3xR3", "Bingham"]
