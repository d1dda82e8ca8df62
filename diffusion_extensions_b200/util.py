"""Drop-in for the SO(3) part of the reference's ``util.py`` (same names, signatures, shapes).

Every function is ONE fused sm_100a kernel on CUDA float32 tensors (via the C ABI in
include/so3d.h); gradients are provided by custom autograd functions whose backward passes are
kernels too.  There is no CPU path.  Reference citations are file:line of
qazwsxal/diffusion-extensions @ f100885d.

Deliberate deviations from the reference (SURVEY.md appendix B):
  * exp maps use the Rodrigues closed form instead of matrix_exp (+ SVD), so results stay
    orthonormal for any scalar (Q5);
  * log_rmat / rmat_to_aa are accurate up to and at a rotation by pi (Q4) and return the axis
    (0,0,1) with angle 0 at the identity instead of NaN (Q10).
"""
import inspect
from collections import namedtuple
from itertools import product
from math import log
from typing import Iterable, Tuple

import torch
import torch.nn.functional as F

from . import ops


# ---------------------------------------------------------------------------------------------
# SE(3) containers (util.py:10-56): a rotation (...,3,3) with a translation (...,3), and the matching
# tangent-space pair the SE(3) denoisers return
# ---------------------------------------------------------------------------------------------
class AffineT(object):
    def __init__(self, rot: torch.Tensor, shift: torch.Tensor):
        super().__init__()
        self.rot = rot
        self.shift = shift

    def __len__(self):
        return max(len(self.rot), len(self.shift))

    def __getitem__(self, item):
        return AffineT(self.rot[item], self.shift[item])

    @property
    def device(self):
        return self.rot.device

    @property
    def shape(self):
        return self.shift.shape

    def to(self, device):
        return AffineT(self.rot.to(device), self.shift.to(device))

    @classmethod
    def from_euler(cls, euls: torch.Tensor, shift: torch.Tensor):
        return cls(euler_to_rmat(*torch.unbind(euls, dim=-1)), shift)

    def detach(self):
        return AffineT(self.rot.detach(), self.shift.detach())

    def clone(self):
        """(not in the reference) a deep copy: what graph-captured steps use for their static input"""
        return AffineT(self.rot.clone(), self.shift.clone())

    def copy_(self, other):
        self.rot.copy_(other.rot)
        self.shift.copy_(other.shift)
        return self


class AffineGrad(object):
    def __init__(self, rot_g, shift_g):
        super().__init__()
        self.rot_g = rot_g
        self.shift_g = shift_g

    def __len__(self):
        return max(len(self.rot_g), len(self.shift_g))

    def __getitem__(self, item):
        return AffineGrad(self.rot_g[item], self.shift_g[item])


def euler_to_rmat(x, y, z):
    """util.py:396-422: R = R_z R_y R_x from the three Euler angles, with the reference's sign convention for
    R_y (its [2,0] entry is +sin y).  Plain torch: data preparation only."""
    cx, sx, cy, sy, cz, sz = torch.cos(x), torch.sin(x), torch.cos(y), -torch.sin(y), torch.cos(z), torch.sin(z)
    rows = (cz * cy, cz * sy * sx - sz * cx, cz * sy * cx + sz * sx,
            sz * cy, sz * sy * sx + cz * cx, sz * sy * cx - cz * sx,
            -sy, cy * sx, cy * cx)
    return torch.stack(rows, dim=-1).reshape(x.shape + (3, 3))


def rmat_to_euler(rmat: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """util.py:388-393."""
    sy = torch.sqrt(rmat[..., 0, 0] * rmat[..., 0, 0] + rmat[..., 1, 0] * rmat[..., 1, 0])
    x = torch.atan2(rmat[..., 2, 1], rmat[..., 2, 2])
    y = torch.atan2(rmat[..., 2, 0], sy)
    z = torch.atan2(rmat[..., 1, 0], rmat[..., 0, 0])
    return x, y, z


# ---------------------------------------------------------------------------------------------
# hat / vee  (util.py:79-92) -- pure data movement, kept as torch indexing (fused away inside the
# kernels wherever they sit on the hot path)
# ---------------------------------------------------------------------------------------------
def rmat2six(x: torch.Tensor) -> torch.Tensor:
    """util.py:62-64: the 6-D rotation representation = the first two ROWS, flattened."""
    return torch.flatten(x[..., :2, :], -2, -1)


def six2rmat(x: torch.Tensor) -> torch.Tensor:
    """util.py:67-76: Gram-Schmidt of the two 3-vectors, third row by the cross product (plain torch: a
    network-output adapter, differentiable, not on the sampling path)."""
    a1, a2 = x[..., :3], x[..., 3:6]
    b1 = a1 / a1.norm(p=2, dim=-1, keepdim=True)
    b2 = a2 - (b1 * a2).sum(dim=-1, keepdim=True) * b1
    b2 = b2 / b2.norm(p=2, dim=-1, keepdim=True)
    return torch.stack((b1, b2, torch.cross(b1, b2, dim=-1)), dim=-2)


def skew2vec(skew: torch.Tensor) -> torch.Tensor:
    return torch.stack((skew[..., 2, 1], -skew[..., 2, 0], skew[..., 1, 0]), dim=-1)


def vec2skew(vec: torch.Tensor) -> torch.Tensor:
    x, y, z = vec[..., 0], vec[..., 1], vec[..., 2]
    o = torch.zeros_like(x)
    return torch.stack((o, -z, y, z, o, -x, -y, x, o), dim=-1).reshape(vec.shape[:-1] + (3, 3))


def orthogonalise(mat):
    """util.py:95-107: U round(S) V^T of the 3x3 block.  Not on the hot path any more (the exp
    maps below are orthonormal by construction); kept for API compatibility."""
    orth_mat = mat.clone()
    u, s, vh = torch.linalg.svd(mat[..., :3, :3])
    orth_mat[..., :3, :3] = u @ torch.diag_embed(s.round()) @ vh
    return orth_mat


# ---------------------------------------------------------------------------------------------
# autograd functions
# ---------------------------------------------------------------------------------------------
class _LogRmat(torch.autograd.Function):
    @staticmethod
    def forward(ctx, r_mat):
        ctx.save_for_backward(r_mat)
        return ops.log_rmat(r_mat)

    @staticmethod
    def backward(ctx, grad):
        (r_mat,) = ctx.saved_tensors
        return ops.log_rmat_bwd(r_mat, grad.contiguous())


class _AaToRmat(torch.autograd.Function):
    @staticmethod
    def forward(ctx, axis, ang):
        # axis (...,3), ang (...,1) already broadcast to a common batch shape
        ctx.save_for_backward(axis, ang)
        return ops.aa_to_rmat(axis, ang[..., 0])

    @staticmethod
    def backward(ctx, grad):
        axis, ang = ctx.saved_tensors
        g_axis, g_ang = ops.aa_to_rmat_bwd(axis.contiguous(), ang[..., 0].contiguous(), grad.contiguous())
        return g_axis, g_ang[..., None]


class _ExpVec(torch.autograd.Function):
    @staticmethod
    def forward(ctx, vec):
        ctx.save_for_backward(vec)
        return ops.exp_vec(vec)

    @staticmethod
    def backward(ctx, grad):
        (vec,) = ctx.saved_tensors
        return ops.exp_vec_bwd(vec.contiguous(), grad.contiguous())


class _So3Scale(torch.autograd.Function):
    @staticmethod
    def forward(ctx, rmat, scalars):
        ctx.save_for_backward(rmat, scalars)
        return ops.so3_scale(rmat, scalars)

    @staticmethod
    def backward(ctx, grad):
        rmat, scalars = ctx.saved_tensors
        bs = torch.broadcast_shapes(rmat.shape[:-2], scalars.shape) if scalars.numel() > 1 else rmat.shape[:-2]
        r = rmat.expand(*bs, 3, 3).contiguous()
        s, stride = ops._per_row(scalars, bs, r.device, "scalars")
        g_r, g_s = ops.so3_scale_bwd(r, s, stride, grad.expand(*bs, 3, 3).contiguous())
        g_r = g_r.sum_to_size(rmat.shape) if g_r.shape != rmat.shape else g_r
        g_s = g_s.sum_to_size(scalars.shape) if g_s.shape != scalars.shape else g_s
        return (g_r if ctx.needs_input_grad[0] else None), (g_s if ctx.needs_input_grad[1] else None)


def _needs_grad(*ts):
    return torch.is_grad_enabled() and any(isinstance(t, torch.Tensor) and t.requires_grad for t in ts)


# ---------------------------------------------------------------------------------------------
# public API (reference names)
# ---------------------------------------------------------------------------------------------
def log_rmat(r_mat: torch.Tensor) -> torch.Tensor:
    """util.py:164-192: matrix logarithm of rotation matrices, (...,3,3) skew-symmetric."""
    if _needs_grad(r_mat):
        return _LogRmat.apply(r_mat)
    return ops.log_rmat(r_mat)


def log_vec(r_mat: torch.Tensor) -> torch.Tensor:
    """skew2vec(log_rmat(R)) in one kernel (the composition used at diffusion.py:355)."""
    if _needs_grad(r_mat):
        return skew2vec(_LogRmat.apply(r_mat))
    return ops.log_vec(r_mat)


def aa_to_rmat(rot_axis: torch.Tensor, ang: torch.Tensor):
    """util.py:195-205: rotation matrix from axis (...,3) (normalised inside) and angle (...,1)."""
    if ang.shape[-1:] != (1,):
        raise ValueError("ang must have a trailing dimension of 1, like the reference (ang[..., None] is applied to it)")
    bs = torch.broadcast_shapes(rot_axis.shape[:-1], ang.shape[:-1])
    if _needs_grad(rot_axis, ang):
        return _AaToRmat.apply(rot_axis.expand(*bs, 3), ang.expand(*bs, 1))
    return ops.aa_to_rmat(rot_axis, ang[..., 0])


def exp_vec(vec: torch.Tensor) -> torch.Tensor:
    """matrix_exp(vec2skew(vec)) (diffusion.py:294) as one kernel."""
    if _needs_grad(vec):
        return _ExpVec.apply(vec)
    return ops.exp_vec(vec)


def rmat_to_aa(r_mat) -> Tuple[torch.Tensor, torch.Tensor]:
    """util.py:208-219: (axis (...,3), angle (...,1)), angle in [0, pi]."""
    if _needs_grad(r_mat):
        skew_vec = skew2vec(_LogRmat.apply(r_mat))
        angle = skew_vec.norm(p=2, dim=-1, keepdim=True)
        # the identity gets the kernel's axis (0,0,1) (Q10); the safe denominator keeps NaN out of the backward too
        nz = angle > 0
        axis = torch.where(nz, skew_vec / torch.where(nz, angle, torch.ones_like(angle)), F.pad(torch.ones_like(angle), (2, 0)))
        return axis, angle
    axis, angle = ops.rmat_to_aa(r_mat)
    return axis, angle[..., None]


def quat_to_rmat(quaternions: torch.Tensor) -> torch.Tensor:
    """util.py:222-252: real-first quaternions (...,4) -> (...,3,3)."""
    if _needs_grad(quaternions):
        r, i, j, k = torch.unbind(quaternions, -1)
        two_s = 2.0 / (quaternions * quaternions).sum(-1)
        o = torch.stack(
            (
                1 - two_s * (j * j + k * k), two_s * (i * j - k * r), two_s * (i * k + j * r),
                two_s * (i * j + k * r), 1 - two_s * (i * i + k * k), two_s * (j * k - i * r),
                two_s * (i * k - j * r), two_s * (j * k + i * r), 1 - two_s * (i * i + j * j),
            ),
            -1,
        )
        return o.reshape(quaternions.shape[:-1] + (3, 3))
    return ops.quat_to_rmat(quaternions)


def rmat_to_quat(r_mat: torch.Tensor) -> torch.Tensor:
    """New (SURVEY D6): unit quaternion (real-first, real part >= 0); inverse of quat_to_rmat."""
    return ops.rmat_to_quat(r_mat)


def rmat_dist(input: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
    """util.py:315-322: geodesic distance as the Frobenius norm of log(input^T target)."""
    if _needs_grad(input, target):
        mul = input.transpose(-1, -2) @ target
        return _LogRmat.apply(mul).norm(p=2, dim=(-1, -2))
    return ops.rmat_dist(input, target)


def so3_lerp(rot_a: torch.Tensor, rot_b: torch.Tensor, weight: torch.Tensor) -> torch.Tensor:
    """util.py:325-338: weight has a trailing dimension of 1 (it multiplies the (...,1) angle)."""
    if _needs_grad(rot_a, rot_b, weight):
        rot_c = rot_a.transpose(-1, -2) @ rot_b
        axis, angle = rmat_to_aa(rot_c)
        return rot_a @ aa_to_rmat(axis, weight * angle)
    w = weight[..., 0] if isinstance(weight, torch.Tensor) and weight.dim() > 0 and weight.shape[-1] == 1 else weight
    return ops.so3_lerp(rot_a, rot_b, w)


def so3_bezier(*rots, weight):
    """util.py:340-346: de Casteljau on SO(3) with so3_lerp.  (The reference recurses with the tuple slices as ONE
    argument, so it only works for two control rotations; this is the evident intent for any number >= 2.)"""
    if len(rots) < 2:
        raise ValueError("so3_bezier needs at least two control rotations")
    if len(rots) == 2:
        return so3_lerp(*rots, weight=weight)
    a = so3_bezier(*rots[:-1], weight=weight)
    b = so3_bezier(*rots[1:], weight=weight)
    return so3_lerp(a, b, weight=weight)


def so3_scale(rmat, scalars):
    """util.py:349-361: scale the rotation angle, exp(scalars * log(rmat))."""
    if not isinstance(scalars, torch.Tensor):
        scalars = torch.tensor(float(scalars), dtype=torch.float32, device=rmat.device)
    if _needs_grad(rmat, scalars):
        return _So3Scale.apply(rmat, scalars)
    return ops.so3_scale(rmat, scalars)


def se3_lerp(transf_a: AffineT, transf_b: AffineT, weight: torch.Tensor) -> AffineT:
    """util.py:364-379: so3_lerp on the rotations, torch.lerp on the translations."""
    return AffineT(so3_lerp(transf_a.rot, transf_b.rot, weight), torch.lerp(transf_a.shift, transf_b.shift, weight))


def se3_scale(transf: AffineT, scalars) -> AffineT:
    """util.py:382-385: so3_scale on the rotation, plain scaling of the translation."""
    return AffineT(so3_scale(transf.rot, scalars), transf.shift * scalars[..., None])


def compose(a, b, trans_a=False, trans_b=False):
    """Batched 3x3 product op(a) @ op(b) as one kernel (no autograd; use `@` when gradients are needed)."""
    return ops.compose(a, b, trans_a, trans_b)


# ---------------------------------------------------------------------------------------------
# kernels on SO(3) and the MMD two-sample statistic  (util.py:108-150, 254-313)
# ---------------------------------------------------------------------------------------------
def rmat_cosine_dist(m1: torch.Tensor, m2: torch.Tensor) -> torch.Tensor:
    """util.py:108-124: 1 - cos(angle of m2^T m1), broadcasting over batch dims."""
    return 1 - rmat_cosine_kernel(m1, m2)


def rmat_gaussian_kernel(m1: torch.Tensor, m2: torch.Tensor) -> torch.Tensor:
    """util.py:128-134: exp(-rmat_dist(m1, m2)), broadcasting over batch dims (one fused distance kernel)."""
    return torch.exp(-rmat_dist(m1, m2))


def rmat_cosine_kernel(m1: torch.Tensor, m2: torch.Tensor) -> torch.Tensor:
    """util.py:136-150: (tr(m2^T m1) - 1) / 2 = cos(angle)."""
    return ((m1 * m2).sum(dim=(-1, -2)) - 1) / 2


_FUSED_PAIR_KERNELS = {rmat_gaussian_kernel: "gaussian", rmat_cosine_kernel: "cosine"}


def MMD(X: torch.Tensor, Y: torch.Tensor, kernel, chunksize=None):
    """util.py:254-285: maximum mean discrepancy between two sets of rotations (biased V-statistic).

    With `rmat_gaussian_kernel` / `rmat_cosine_kernel` the three all-pairs sums run as ONE fused sm_100a launch that
    never materialises a pair matrix (so `chunksize`, the reference's memory workaround, is not needed and is
    ignored); any other callable takes the reference's chunked outer-product route through torch ops."""
    l_X, l_Y = len(X), len(Y)
    fused = _FUSED_PAIR_KERNELS.get(kernel)
    if fused is not None and X.is_cuda and X.dim() == 3 and Y.dim() == 3 and not _needs_grad(X, Y):
        sums = ops.pair_kernel_sums(X, Y, fused)
        mmd = sums[0] / (l_X ** 2) + sums[1] / (l_Y ** 2) - sums[2] * (2 / (l_X * l_Y))
        return mmd.to(torch.float32)
    maxlen = max(l_X, l_Y)
    if chunksize is None or chunksize >= maxlen:
        X_sum = kernel(X.unsqueeze(0), X.unsqueeze(1)).sum(dim=(0, 1))
        Y_sum = kernel(Y.unsqueeze(0), Y.unsqueeze(1)).sum(dim=(0, 1))
        XY_sum = kernel(X.unsqueeze(0), Y.unsqueeze(1)).sum(dim=(0, 1))
    else:
        splits = list(range(chunksize, maxlen, chunksize))
        X_split = torch.tensor_split(X, splits)
        Y_split = torch.tensor_split(Y, splits)
        X_sum = sum(kernel(x1.unsqueeze(0), x2.unsqueeze(1)).sum(dim=(0, 1)) for x1, x2 in product(X_split, X_split))
        Y_sum = sum(kernel(y1.unsqueeze(0), y2.unsqueeze(1)).sum(dim=(0, 1)) for y1, y2 in product(Y_split, Y_split))
        XY_sum = sum(kernel(x.unsqueeze(0), y.unsqueeze(1)).sum(dim=(0, 1)) for x, y in product(X_split, Y_split))
    return (1 / (l_X ** 2)) * X_sum + (1 / (l_Y ** 2)) * Y_sum - (2 / (l_X * l_Y)) * XY_sum


def Ker_2samp_test(X, Y, kernel, alpha=0.05, max_ker=1, chunksize=None):
    """util.py:287-298: kernel two-sample test (True = same distribution not rejected)."""
    m, n = len(X), len(Y)
    assert m == n, "Requires equal amount of samples from X and Y"
    mmd = MMD(X, Y, kernel, chunksize=chunksize).item()
    test_val = (2 * max_ker / m) ** 0.5 * (1 + (2 * log(1 / alpha)) ** 0.5)
    return mmd < test_val


def Ker_2samp_log_prob(X, Y, kernel, max_ker=1, chunksize=None):
    """util.py:300-312: log-probability of a type I error."""
    m, n = len(X), len(Y)
    assert m == n, "Requires equal amount of samples from X and Y"
    mmd = MMD(X, Y, kernel, chunksize=chunksize).item()
    return -((((mmd / ((2 * max_ker / m) ** 0.5)) - 1) ** 2) / 2)


__all__ = [
    "skew2vec", "vec2skew", "orthogonalise", "log_rmat", "log_vec", "aa_to_rmat", "exp_vec", "rmat_to_aa",
    "quat_to_rmat", "rmat_to_quat", "rmat_dist", "so3_lerp", "so3_scale", "compose",
    "AffineT", "AffineGrad", "euler_to_rmat", "rmat_to_euler", "se3_lerp", "se3_scale",
    "rmat_cosine_dist", "rmat_gaussian_kernel", "rmat_cosine_kernel", "MMD", "Ker_2samp_test", "Ker_2samp_log_prob",
]


# ---------------------------------------------------------------------------------------------
# small helpers the reference's scripts import from util (util.py:59, 426-481).  REFERENCE-DERIVED API SHIMS, not part
# of the hot path: `from util import *` in the reference's scripts pulls these names in, so they are restated here
# (same names, arguments and behaviour; plain host-side Python, no kernels).  The same holds for the `AffineT` /
# `AffineGrad` containers at the top of this file (util.py:10-56): their attribute surface IS the interface.
# ---------------------------------------------------------------------------------------------
ProtData = namedtuple("ProtData", ["residues", "positions", "angles"])  # util.py:59 (the docking scripts' batch record)


def to_device(device, *objects, non_blocking=False):
    """util.py:426-437: move tensors / AffineT / ProtData / nested iterables of them to `device`, keeping the structure
    (a ProtData comes back as a ProtData, like the reference)."""
    out = []
    for obj in objects:
        if isinstance(obj, (torch.Tensor, AffineT)):
            out.append(obj.to(device, non_blocking=non_blocking) if isinstance(obj, torch.Tensor) else obj.to(device))
        elif isinstance(obj, ProtData):
            out.append(ProtData(*to_device(device, *obj, non_blocking=non_blocking)))
        elif isinstance(obj, Iterable) and not isinstance(obj, (str, bytes)):
            out.append(to_device(device, *obj, non_blocking=non_blocking))
        else:
            raise NotImplementedError(f"Object type {type(obj)} unsupported")
    return out


def init_from_dict(argdict, *classes):
    """util.py:440-460: build each class from the entries of `argdict` its constructor names (others ignored)."""
    objs = []
    for cls in classes:
        names = [k for k, v in inspect.signature(cls).parameters.items() if v.kind == inspect.Parameter.POSITIONAL_OR_KEYWORD]
        objs.append(cls(**{k: v for k, v in argdict.items() if k in names}))
    return objs


def identity(x):
    return x


def masked_mean(tensor, mask, dim=-1):
    """util.py:467-475: mean over `dim` of the entries where mask is set (0 where none are); zeroes the masked
    entries of `tensor` IN PLACE like the reference."""
    mask = mask[(..., *((None,) * (tensor.dim() - mask.dim())))]
    tensor.masked_fill_(~mask, 0.)
    total = mask.sum(dim=dim)
    mean = tensor.sum(dim=dim) / total.clamp(min=1.)
    mean.masked_fill_(total == 0, 0.)
    return mean


def cycle(iterable):
    """util.py:478-481: endless iterator over `iterable` (restarts it when exhausted)."""
    while True:
        for x in iterable:
            yield x
