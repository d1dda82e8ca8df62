"""Tensor-level wrappers over the C ABI (no autograd here; see util.py / distributions.py).

Every function takes CUDA float32 tensors with arbitrary leading batch dims, flattens them to
rows, launches ONE fused kernel on the current stream and returns freshly allocated tensors.
Nothing here synchronises with the host.
"""
import math

import torch

from . import _lib
from ._lib import call, check_f32, ptr

CDF_POINTS = 999
GRID_POINTS = 1000
GUIDE_BUCKETS = 2051  # 16-byte records per guide row (include/so3d.h SO3D_GUIDE_BUCKETS)


# ---------------------------------------------------------------------------------------------
# counter-based RNG state (Philox key/offset), following torch.manual_seed like a torch op would
# ---------------------------------------------------------------------------------------------
class _Rng:
    """(seed, offset) of every sampling launch.

    Two regimes:
      * after ``dx.manual_seed(s)``: an explicit stream -- seed s, offsets 0, 1, 2, ... (one per launch) -- until
        ``torch.manual_seed`` installs a different seed;
      * otherwise the launches FOLLOW TORCH'S CUDA GENERATOR like any torch op: the seed is the generator's seed and
        the offset is its Philox offset, which the launch advances by 4 (one Philox block per row).  ``torch.manual_seed(s)``
        therefore resets the stream even when s equals the previous seed (the usual way to reproduce a run), and the
        draws interleave deterministically with torch's own random ops.
    While a CUDA graph is being captured the generator's offset cannot be touched from the host; captured launches read
    their seed from device memory instead (`use_device_seed`, `*_dseed_f32`) and never come through here."""

    def __init__(self):
        self.seed = None
        self.offset = 0
        self._torch_seed = None
        self._explicit = False

    def manual_seed(self, seed):
        self.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        self.offset = 0
        self._torch_seed = torch.initial_seed()
        self._explicit = True

    def next(self, device=None):
        """(seed, offset) for one sampling launch; every launch gets a fresh offset."""
        ts = torch.initial_seed()
        if self._explicit and ts == self._torch_seed:
            off = self.offset
            self.offset += 1
            return self.seed, off
        self._explicit = False
        if torch.cuda.is_available() and not torch.cuda.is_current_stream_capturing():
            idx = torch.cuda.current_device() if device is None or torch.device(device).index is None else torch.device(device).index
            gen = torch.cuda.default_generators[idx]
            off = int(gen.get_offset())
            gen.set_offset(off + 4)
            self.seed, self.offset, self._torch_seed = int(gen.initial_seed()) & 0xFFFFFFFFFFFFFFFF, off // 4 + 1, ts
            return self.seed, off // 4
        # no CUDA generator to follow (CPU-only unit tests of the host logic) or inside a capture: private counter
        if self.seed is None or ts != self._torch_seed:
            self.seed, self.offset, self._torch_seed = ts & 0xFFFFFFFFFFFFFFFF, 0, ts
        off = self.offset
        self.offset += 1
        return self.seed, off


rng = _Rng()


def manual_seed(seed):
    """Seed an explicit Philox stream for the sampling kernels (offsets 0, 1, 2, ... per launch).  Without it the
    kernels follow torch's CUDA generator, so ``torch.manual_seed(s)`` -- with a new OR the same s -- resets them too."""
    rng.manual_seed(seed)


# ---------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------
def _rows9(x, name):
    x = check_f32(x, name, (3, 3))
    return x, x.shape[:-2], x.numel() // 9


def _rows3(x, name):
    x = check_f32(x, name, (3,))
    return x, x.shape[:-1], x.numel() // 3


def _per_row(s, batch_shape, device, name):
    """Per-row scalar operand -> (tensor, stride): stride 0 for a single shared value."""
    if not isinstance(s, torch.Tensor):
        s = torch.tensor(float(s), dtype=torch.float32, device=device)
    s = check_f32(s, name)
    if s.numel() == 1:
        return s.reshape(1), 0
    s = s.expand(batch_shape).contiguous() if tuple(s.shape) != tuple(batch_shape) else s
    return s, 1


def _bcast2(a, b):
    """Broadcast the batch dims of two (...,3,3) tensors."""
    if a.shape != b.shape:
        bs = torch.broadcast_shapes(a.shape[:-2], b.shape[:-2])
        a = a.expand(*bs, 3, 3).contiguous()
        b = b.expand(*bs, 3, 3).contiguous()
    return a, b


# ---------------------------------------------------------------------------------------------
# L0
# ---------------------------------------------------------------------------------------------
def log_rmat(R):
    R, bs, n = _rows9(R, "r_mat")
    out = torch.empty_like(R)
    call("so3d_log_f32", ptr(R), ptr(out), n, device=R.device)
    return out


def log_vec(R):
    R, bs, n = _rows9(R, "r_mat")
    out = torch.empty(*bs, 3, dtype=torch.float32, device=R.device)
    call("so3d_logvec_f32", ptr(R), ptr(out), n, device=R.device)
    return out


def rmat_to_aa(R):
    """-> unit axis (...,3), angle (...)"""
    R, bs, n = _rows9(R, "r_mat")
    axis = torch.empty(*bs, 3, dtype=torch.float32, device=R.device)
    angle = torch.empty(*bs, dtype=torch.float32, device=R.device)
    call("so3d_rmat_to_aa_f32", ptr(R), ptr(axis), ptr(angle), n, device=R.device)
    return axis, angle


def aa_to_rmat(axis, angle):
    """axis (...,3) (normalised inside), angle (...)"""
    axis = check_f32(axis, "rot_axis", (3,))
    angle = check_f32(angle, "ang")
    bs = torch.broadcast_shapes(axis.shape[:-1], angle.shape)
    axis = axis.expand(*bs, 3).contiguous()
    angle = angle.expand(bs).contiguous()
    out = torch.empty(*bs, 3, 3, dtype=torch.float32, device=axis.device)
    call("so3d_aa_to_rmat_f32", ptr(axis), ptr(angle), ptr(out), angle.numel(), device=axis.device)
    return out


def exp_vec(v):
    v, bs, n = _rows3(v, "vec")
    out = torch.empty(*bs, 3, 3, dtype=torch.float32, device=v.device)
    call("so3d_expvec_f32", ptr(v), ptr(out), n, device=v.device)
    return out


def so3_scale(R, scalars):
    R = check_f32(R, "rmat", (3, 3))
    if isinstance(scalars, torch.Tensor) and scalars.numel() > 1 and tuple(scalars.shape) != tuple(R.shape[:-2]):
        bs = torch.broadcast_shapes(R.shape[:-2], scalars.shape)
        R = R.expand(*bs, 3, 3).contiguous()
    bs, n = R.shape[:-2], R.numel() // 9
    s, stride = _per_row(scalars, bs, R.device, "scalars")
    out = torch.empty_like(R)
    call("so3d_scale_f32", ptr(R), ptr(s), stride, ptr(out), n, device=R.device)
    return out


def quat_to_rmat(q):
    q = check_f32(q, "quaternions", (4,))
    out = torch.empty(*q.shape[:-1], 3, 3, dtype=torch.float32, device=q.device)
    call("so3d_quat_to_rmat_f32", ptr(q), ptr(out), q.numel() // 4, device=q.device)
    return out


def rmat_to_quat(R):
    R, bs, n = _rows9(R, "r_mat")
    out = torch.empty(*bs, 4, dtype=torch.float32, device=R.device)
    call("so3d_rmat_to_quat_f32", ptr(R), ptr(out), n, device=R.device)
    return out


def compose(A, B, trans_a=False, trans_b=False):
    """op(A) @ op(B) for batched 3x3; a single (3,3) operand is shared by all rows."""
    A = check_f32(A, "A", (3, 3))
    B = check_f32(B, "B", (3, 3))
    if A.numel() == 9 and B.numel() > 9:
        sa, sb, bs, n = 0, 1, B.shape[:-2], B.numel() // 9
    elif B.numel() == 9 and A.numel() > 9:
        sa, sb, bs, n = 1, 0, A.shape[:-2], A.numel() // 9
    else:
        A, B = _bcast2(A, B)
        sa, sb, bs, n = 1, 1, A.shape[:-2], A.numel() // 9
    out = torch.empty(*bs, 3, 3, dtype=torch.float32, device=A.device)
    call("so3d_compose_f32", ptr(A), sa, int(trans_a), ptr(B), sb, int(trans_b), ptr(out), n, device=A.device)
    return out


def rmat_dist(A, B):
    A = check_f32(A, "input", (3, 3))
    B = check_f32(B, "target", (3, 3))
    A, B = _bcast2(A, B)
    out = torch.empty(A.shape[:-2], dtype=torch.float32, device=A.device)
    call("so3d_rmat_dist_f32", ptr(A), ptr(B), ptr(out), A.numel() // 9, device=A.device)
    return out


def so3_lerp(A, B, weight):
    """weight: (...) (no trailing 1)."""
    A = check_f32(A, "rot_a", (3, 3))
    B = check_f32(B, "rot_b", (3, 3))
    A, B = _bcast2(A, B)
    w, stride = _per_row(weight, A.shape[:-2], A.device, "weight")
    out = torch.empty_like(A)
    call("so3d_lerp_f32", ptr(A), ptr(B), ptr(w), stride, ptr(out), A.numel() // 9, device=A.device)
    return out


# backward passes
def log_rmat_bwd(R, G):
    R, _, n = _rows9(R, "r_mat")
    G = check_f32(G, "grad", (3, 3))
    out = torch.empty_like(R)
    call("so3d_log_bwd_f32", ptr(R), ptr(G), ptr(out), n, device=R.device)
    return out


def aa_to_rmat_bwd(axis, angle, G):
    axis = check_f32(axis, "rot_axis", (3,))
    angle = check_f32(angle, "ang")
    G = check_f32(G, "grad", (3, 3))
    g_axis = torch.empty_like(axis)
    g_angle = torch.empty_like(angle)
    call("so3d_aa_to_rmat_bwd_f32", ptr(axis), ptr(angle), ptr(G), ptr(g_axis), ptr(g_angle), angle.numel(), device=axis.device)
    return g_axis, g_angle


def exp_vec_bwd(v, G):
    v = check_f32(v, "vec", (3,))
    G = check_f32(G, "grad", (3, 3))
    out = torch.empty_like(v)
    call("so3d_expvec_bwd_f32", ptr(v), ptr(G), ptr(out), v.numel() // 3, device=v.device)
    return out


def so3_scale_bwd(R, s, stride, G):
    """-> grad wrt R (...,3,3), per-row grad wrt the scalar (...)"""
    R, bs, n = _rows9(R, "rmat")
    G = check_f32(G, "grad", (3, 3))
    gR = torch.empty_like(R)
    gs = torch.empty(bs, dtype=torch.float32, device=R.device)
    call("so3d_scale_bwd_f32", ptr(R), ptr(s), stride, ptr(G), ptr(gR), ptr(gs), n, device=R.device)
    return gR, gs


# ---------------------------------------------------------------------------------------------
# L1: IGSO(3)
# ---------------------------------------------------------------------------------------------
def _mode(mode):
    if isinstance(mode, str):
        if mode not in _lib.MODES:
            raise ValueError(f"mode must be one of {sorted(_lib.MODES)}")
        return _lib.MODES[mode]
    return int(mode)


def igso3_density(omega, eps, mode="closed", L=2000):
    omega = check_f32(omega, "t")
    eps_t, stride = _per_row(eps, omega.shape, omega.device, "eps")
    out = torch.empty_like(omega)
    call("so3d_igso3_density_f32", ptr(omega), ptr(eps_t), stride, ptr(out), omega.numel(), _mode(mode), int(L), device=omega.device)
    return out


def igso3_logp_score(R, eps, mode="auto", L=2000, want_score=True, want_dlogf=False):
    """-> logp (...), score (...,3) or None, dlogf (...) or None"""
    R, bs, n = _rows9(R, "rotations")
    eps_t, stride = _per_row(eps, bs, R.device, "eps")
    logp = torch.empty(bs, dtype=torch.float32, device=R.device)
    score = torch.empty(*bs, 3, dtype=torch.float32, device=R.device) if want_score else None
    dlogf = torch.empty(bs, dtype=torch.float32, device=R.device) if want_dlogf else None
    call("so3d_igso3_logp_score_f32", ptr(R), ptr(eps_t), stride, ptr(logp), ptr(score), ptr(dlogf), n, _mode(mode), int(L), device=R.device)
    return logp, score, dlogf


def igso3_logp_bwd(R, dlogf, gout):
    R, bs, n = _rows9(R, "rotations")
    dlogf = check_f32(dlogf, "dlogf")
    gout = check_f32(gout.expand(bs), "grad_output")
    out = torch.empty_like(R)
    call("so3d_igso3_logp_bwd_f32", ptr(R), ptr(dlogf), ptr(gout), ptr(out), n, device=R.device)
    return out


class HostScorePipeline:
    """Streams HOST (pinned) rotations / eps through the fused log-density + score kernel and returns HOST
    results, overlapping the three legs chunk by chunk on separate CUDA streams:

        H2D copy of chunk k+1   ||   kernel on chunk k   ||   D2H copy of the results of chunk k-1

    With 40 B in and 16 B out per evaluation the PCIe link (not the kernel) bounds the end-to-end rate, so the
    pipeline runs at the speed of the slowest leg instead of their sum.  Device staging buffers are a ring of
    `depth` chunks allocated once; nothing synchronises with the host until `run` returns (it waits for the
    last D2H copy, because the caller is about to read host memory).

    Streaming several batches: `run(..., wait=False, join=False)` neither joins the pipeline's streams to the current
    stream at entry nor at exit, so the H2D copies of the next batch start while the previous batch's last kernels and
    D2H copies drain (the staging slots are guarded by events that persist across calls); call `finish()` once at the
    end to make the current stream wait for everything issued so far."""

    def __init__(self, device, chunk_rows=1 << 20, depth=3, per_row_eps=True):
        self.device = torch.device(device)
        self.chunk, self.depth = int(chunk_rows), int(depth)
        d = self.device
        self.dR = [torch.empty(self.chunk, 3, 3, device=d) for _ in range(depth)]
        self.deps = [torch.empty(self.chunk, device=d) for _ in range(depth)] if per_row_eps else None
        self.dlogp = [torch.empty(self.chunk, device=d) for _ in range(depth)]
        self.dscore = [torch.empty(self.chunk, 3, device=d) for _ in range(depth)]
        self.s_in, self.s_k, self.s_out = (torch.cuda.Stream(d) for _ in range(3))
        self.ev_in = [torch.cuda.Event() for _ in range(depth)]
        self.ev_k = [torch.cuda.Event() for _ in range(depth)]
        self.ev_out = [torch.cuda.Event() for _ in range(depth)]
        self.launches = 0
        self.issued = 0  # chunks issued so far over all calls: slot b has been used before iff issued > b

    def finish(self, wait=False):
        """Make the current stream wait for every chunk issued so far (and optionally the host too)."""
        cur = torch.cuda.current_stream(self.device)
        cur.wait_stream(self.s_out)
        cur.wait_stream(self.s_k)
        if wait:
            self.s_out.synchronize()

    def run(self, hR, heps, h_logp, h_score, mode="series", L=2000, wait=True, join=True):
        """hR (n,3,3), heps (n,) or a scalar tensor/float, h_logp (n,), h_score (n,3): pinned host float32 tensors."""
        for name, t in (("rotations", hR), ("logp", h_logp), ("score", h_score)):
            if t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous():
                raise ValueError(f"{name} must be a contiguous float32 HOST tensor")
        n = hR.shape[0]
        per_row = isinstance(heps, torch.Tensor) and heps.numel() == n and n > 1
        if per_row and self.deps is None:
            raise ValueError("pipeline was created with per_row_eps=False")
        eps_shared = None if per_row else torch.as_tensor(heps, dtype=torch.float32).reshape(1).to(self.device)
        m = _mode(mode)
        cur = torch.cuda.current_stream(self.device)
        if join:
            for st in (self.s_in, self.s_k, self.s_out):
                st.wait_stream(cur)
        if eps_shared is not None:
            self.s_k.wait_stream(cur)                       # the shared eps was uploaded on the current stream
        for lo in range(0, n, self.chunk):
            hi = min(n, lo + self.chunk)
            rows, b = hi - lo, self.issued % self.depth
            used = self.issued >= self.depth                # the slot carries a chunk of this or an earlier call
            self.issued += 1
            with torch.cuda.stream(self.s_in):
                if used:
                    self.s_in.wait_event(self.ev_k[b])      # the kernel that read this staging slot is done
                self.dR[b][:rows].copy_(hR[lo:hi], non_blocking=True)
                if per_row:
                    self.deps[b][:rows].copy_(heps[lo:hi], non_blocking=True)
                self.ev_in[b].record(self.s_in)
            with torch.cuda.stream(self.s_k):
                self.s_k.wait_event(self.ev_in[b])
                if used:
                    self.s_k.wait_event(self.ev_out[b])     # the D2H copy that read this result slot is done
                e = self.deps[b] if per_row else eps_shared
                call("so3d_igso3_logp_score_f32", ptr(self.dR[b]), ptr(e), 1 if per_row else 0, ptr(self.dlogp[b]), ptr(self.dscore[b]), None,
                     rows, m, int(L), device=self.device)
                self.launches += 1
                self.ev_k[b].record(self.s_k)
            with torch.cuda.stream(self.s_out):
                self.s_out.wait_event(self.ev_k[b])
                h_logp[lo:hi].copy_(self.dlogp[b][:rows], non_blocking=True)
                h_score[lo:hi].copy_(self.dscore[b][:rows], non_blocking=True)
                self.ev_out[b].record(self.s_out)
        if join or wait:
            self.finish(wait=wait)
        return h_logp, h_score


_grid_cache = {}


def cdf_grid(device):
    """The reference's 1000-point float32 grid and Haar weights, computed with the same torch CPU
    ops the reference uses (distributions.py:15, :21) so the float32 values are bit-identical.
    -> (grid_loc[1000], haar_w[1000], trap_loc[999]) on `device`."""
    key = str(device)
    if key not in _grid_cache:
        loc = math.pi * torch.linspace(0, 1.0, GRID_POINTS) ** 3.0
        haar = (1 - loc.cos()) / math.pi
        loc_d = loc.to(device)
        _grid_cache[key] = (loc_d, haar.to(device), loc_d[1:].contiguous())
    return _grid_cache[key]


def igso3_cdf_table(eps, reference_quirks=False):
    """eps (rows,) -> trap (rows, 999): one CDF row per eps (distributions.py:15-30)."""
    eps = check_f32(eps, "eps").reshape(-1)
    loc, haar, _ = cdf_grid(eps.device)
    out = torch.empty(eps.numel(), CDF_POINTS, dtype=torch.float32, device=eps.device)
    call("so3d_igso3_cdf_table_f32", ptr(eps), eps.numel(), ptr(loc), ptr(haar), ptr(out), int(bool(reference_quirks)), device=eps.device)
    return out


def igso3_cdf_guide(cdf):
    """cdf (rows, 999) -> guide (rows, 2051, 4) int32: the 16-byte search records of include/so3d.h."""
    cdf = check_f32(cdf, "cdf", (CDF_POINTS,))
    rows = cdf.numel() // CDF_POINTS
    out = torch.empty(rows, GUIDE_BUCKETS, 4, dtype=torch.int32, device=cdf.device)
    call("so3d_igso3_cdf_guide", ptr(cdf), rows, ptr(out), device=cdf.device)
    return out


def _check_guide(guide, rows, name):
    if guide is not None and (guide.dtype != torch.int32 or guide.numel() != rows * GUIDE_BUCKETS * 4 or not guide.is_contiguous() or not guide.is_cuda):
        raise ValueError(f"{name} must be the contiguous CUDA int32 (rows, {GUIDE_BUCKETS}, 4) tensor returned by igso3_cdf_guide")
    return guide


def igso3_sample(cdf, shape, row_idx=None, row=0, u=None, axes=None, seed=None, rng_offset=None, row_offset=0,
                 mean=None, want_angle=False, want_axis=False, guide=None):
    """Draw rotations of batch shape `shape` from the CDF rows in `cdf` (rows, 999).
    row_idx: int64 tensor of shape `shape` (one table row per sample) or None -> all use `row`.
    u / axes: optional explicit draws.  -> R (*shape,3,3)[, angle (*shape)][, axis (*shape,3)]"""
    cdf = check_f32(cdf, "cdf", (CDF_POINTS,))
    dev = cdf.device
    shape = tuple(shape)
    n = 1
    for d in shape:
        n *= int(d)
    _, _, trap_loc = cdf_grid(dev)
    if row_idx is not None:
        row_idx = row_idx.to(device=dev, dtype=torch.int64).expand(shape).contiguous()
    if u is not None:
        u = check_f32(u, "u").expand(shape).contiguous()
    if axes is not None:
        axes = check_f32(axes, "axes", (3,)).expand(*shape, 3).contiguous()
    if seed is None or rng_offset is None:
        seed, rng_offset = rng.next()
    mean_stride = 0
    if mean is not None:
        mean = check_f32(mean, "mean", (3, 3))
        if mean.numel() != 9:
            mean = mean.expand(*shape, 3, 3).contiguous()
            mean_stride = 1
    R = torch.empty(*shape, 3, 3, dtype=torch.float32, device=dev)
    angle = torch.empty(shape, dtype=torch.float32, device=dev) if want_angle else None
    axis_out = torch.empty(*shape, 3, dtype=torch.float32, device=dev) if want_axis else None
    _check_guide(guide, cdf.numel() // CDF_POINTS, "guide")
    call("so3d_igso3_sample_f32", ptr(cdf), ptr(guide), ptr(trap_loc), cdf.numel() // CDF_POINTS, ptr(row_idx), int(row), ptr(u), ptr(axes),
         seed, rng_offset, int(row_offset), ptr(mean), mean_stride, ptr(R), ptr(angle), ptr(axis_out), n, device=dev)
    outs = [R]
    if want_angle:
        outs.append(angle)
    if want_axis:
        outs.append(axis_out)
    return outs[0] if len(outs) == 1 else tuple(outs)


def igso3_sample_exact(eps, shape, u=None, axes=None, seed=None, rng_offset=None, row_offset=0, mean=None,
                       want_angle=False, want_axis=False):
    """Draw rotations of batch shape `shape` from IGSO(3)(eps) with the angle from the exact inverse CDF of the angle law
    (no CDF table: per-row eps costs one float per row).  eps: a scalar / one-element tensor, or a tensor that broadcasts
    to `shape` (one eps per sample).  u / axes / seed / rng_offset / row_offset / mean as in `igso3_sample`, with the same
    Philox counter layout: at the same (seed, rng_offset, row_offset) both samplers draw the same (u, axis).
    -> R (*shape,3,3)[, angle (*shape)][, axis (*shape,3)]"""
    shape = tuple(shape)
    if isinstance(eps, torch.Tensor):
        dev = eps.device
    else:
        dev = torch.device("cuda", torch.cuda.current_device())
    n = 1
    for d in shape:
        n *= int(d)
    eps_t, eps_stride = _per_row(eps, shape, dev, "eps")
    if u is not None:
        u = check_f32(u, "u").expand(shape).contiguous()
    if axes is not None:
        axes = check_f32(axes, "axes", (3,)).expand(*shape, 3).contiguous()
    if seed is None or rng_offset is None:
        seed, rng_offset = rng.next()
    mean_stride = 0
    if mean is not None:
        mean = check_f32(mean, "mean", (3, 3))
        if mean.numel() != 9:
            mean = mean.expand(*shape, 3, 3).contiguous()
            mean_stride = 1
    R = torch.empty(*shape, 3, 3, dtype=torch.float32, device=dev)
    angle = torch.empty(shape, dtype=torch.float32, device=dev) if want_angle else None
    axis_out = torch.empty(*shape, 3, dtype=torch.float32, device=dev) if want_axis else None
    call("so3d_igso3_sample_exact_f32", ptr(eps_t), eps_stride, ptr(u), ptr(axes), seed, rng_offset, int(row_offset), ptr(mean),
         mean_stride, ptr(R), ptr(angle), ptr(axis_out), n, device=dev)
    outs = [R]
    if want_angle:
        outs.append(angle)
    if want_axis:
        outs.append(axis_out)
    return outs[0] if len(outs) == 1 else tuple(outs)


def igso3_entropy(eps, want_grad=False):
    """Entropy of IGSO(3)(eps) w.r.t. normalised Haar measure and its eps-derivative (de Bruijn: 2 eps E[(d log f / dw)^2]).
    eps: float32 CUDA tensor of any shape.  -> (H, dH/deps or None), both shaped like eps."""
    e = check_f32(eps, "eps")
    H = torch.empty_like(e)
    dH = torch.empty_like(e) if want_grad else None
    call("so3d_igso3_entropy_f32", ptr(e), ptr(H), ptr(dH), e.numel(), device=e.device)
    return H, dH


def igso3_rsample_bwd(eps, angle, axis, G, u=None, seed=0, rng_offset=0, row_offset=0, mean=None, want_mean_grad=True):
    """Backward of `igso3_sample_exact` read as a reparameterised draw R = mean exp(angle hat(axis)), angle = F^{-1}(u; eps)
    at fixed (u, axis).  angle (*shape) / axis (*shape,3): the forward's outputs; G (*shape,3,3): dL/dR.  eps / u / seed /
    rng_offset / row_offset / mean as the forward got them (u and the Philox stream are read only at rows where eps == 0,
    whose derivative is the eps -> 0+ limit 2 x0(u)).
    -> (g_eps (*shape): dL/deps per row -- reduce it for a shared eps --, g_mean (*shape,3,3) = G N^T per row, or None)"""
    shape = tuple(angle.shape)
    dev = angle.device
    n = angle.numel()
    angle = check_f32(angle, "angle").contiguous()
    axis = check_f32(axis, "axis", (3,)).expand(*shape, 3).contiguous()
    G = check_f32(G, "G", (3, 3)).expand(*shape, 3, 3).contiguous()
    eps_t, eps_stride = _per_row(eps, shape, dev, "eps")
    if u is not None:
        u = check_f32(u, "u").expand(shape).contiguous()
    mean_stride = 0
    if mean is not None:
        mean = check_f32(mean, "mean", (3, 3))
        if mean.numel() != 9:
            mean = mean.expand(*shape, 3, 3).contiguous()
            mean_stride = 1
        else:
            mean = mean.contiguous()
    g_eps = torch.empty(shape, dtype=torch.float32, device=dev)
    g_mean = torch.empty(*shape, 3, 3, dtype=torch.float32, device=dev) if want_mean_grad else None
    call("so3d_igso3_rsample_bwd_f32", ptr(eps_t), eps_stride, ptr(angle), ptr(axis), ptr(mean), mean_stride, ptr(G), ptr(u),
         int(seed), int(rng_offset), int(row_offset), ptr(g_eps), ptr(g_mean), n, device=dev)
    return g_eps, g_mean


# ---------------------------------------------------------------------------------------------
# SE(3) arm: fused forward noising / reverse step on (rotation, translation) pairs (diffusion.py:432-573)
# ---------------------------------------------------------------------------------------------
def _rows_t(t, bs, dev):
    """t (int64) broadcast against the batch shape `bs`: leading dims are matched first, like the reference's
    extract(a, t, t.shape)[..., None] broadcasting of a (B,) step index over (B, N_res, ...) frames."""
    t = t.to(device=dev, dtype=torch.int64)
    if tuple(t.shape) != tuple(bs):
        t = t.reshape(tuple(t.shape) + (1,) * (len(bs) - t.dim())).expand(bs)
    return t.contiguous()


def se3_q_sample_fused(rot0, shift0, t, sqrt_ac, sqrt_1m_ac, cdf, shift_scale, seed=None, rng_offset=None, row_offset=0,
                       want_target=True, guide=None):
    """-> dict(rot, shift, target_rot, target_shift).  seed: an int with rng_offset (by value), None (the module's Philox
    stream), or a one-element int64 device tensor read when the kernel runs (CUDA-graph replays; rng_offset required)."""
    rot0, bs, n = _rows9(rot0, "x_start.rot")
    dev = rot0.device
    shift0 = check_f32(shift0, "x_start.shift", (3,)).expand(*bs, 3).contiguous()
    t = _rows_t(t, bs, dev)
    sqrt_ac = check_f32(sqrt_ac, "sqrt_alphas_cumprod")
    sqrt_1m_ac = check_f32(sqrt_1m_ac, "sqrt_one_minus_alphas_cumprod")
    cdf = check_f32(cdf, "cdf", (CDF_POINTS,))
    T = sqrt_ac.numel()
    if cdf.numel() != T * CDF_POINTS:
        raise ValueError("cdf table must have one row per timestep")
    _check_guide(guide, T, "guide")
    _, _, trap_loc = cdf_grid(dev)
    seed_dev = _seed_tensor(seed, dev)
    if seed_dev is not None and rng_offset is None:
        raise ValueError("a device seed needs an explicit rng_offset")
    if seed_dev is None and (seed is None or rng_offset is None):
        seed, rng_offset = rng.next()
    rot_t, shift_t = torch.empty_like(rot0), torch.empty_like(shift0)
    tr = torch.empty_like(shift0) if want_target else None
    ts = torch.empty_like(shift0) if want_target else None
    if seed_dev is not None:  # CUDA-graph replayable launch: the seed is read on the device when the kernel runs
        call("so3d_se3_q_sample_dseed_f32", ptr(rot0), ptr(shift0), ptr(t), ptr(sqrt_ac), ptr(sqrt_1m_ac), T, ptr(cdf), ptr(guide), ptr(trap_loc),
             float(shift_scale), ptr(seed_dev), int(rng_offset), int(row_offset), ptr(rot_t), ptr(shift_t), ptr(tr), ptr(ts), n, device=dev)
        return {"rot": rot_t, "shift": shift_t, "target_rot": tr, "target_shift": ts}
    call("so3d_se3_q_sample_f32", ptr(rot0), ptr(shift0), ptr(t), ptr(sqrt_ac), ptr(sqrt_1m_ac), T, ptr(cdf), ptr(guide), ptr(trap_loc),
         float(shift_scale), seed, rng_offset, int(row_offset), ptr(rot_t), ptr(shift_t), ptr(tr), ptr(ts), n, device=dev)
    return {"rot": rot_t, "shift": shift_t, "target_rot": tr, "target_shift": ts}


def se3_p_sample_fused(rot_t, shift_t, pred_rot, pred_shift, t, recip, recipm1, coef1, coef2, sigma, shift_scale, post_cdf=None,
                       seed=None, rng_offset=None, row_offset=0, post_guide=None):
    """Fused SE(3) reverse step; t with one element = shared step.  post_cdf None -> posterior mean only.
    seed may be a one-element int64 device tensor read when the kernel runs (CUDA-graph replays): that takes a shared
    step, post_cdf and an explicit rng_offset.  -> (rot (...,3,3), shift (...,3))"""
    rot_t, bs, n = _rows9(rot_t, "x.rot")
    dev = rot_t.device
    shift_t = check_f32(shift_t, "x.shift", (3,)).expand(*bs, 3).contiguous()
    pred_rot = check_f32(pred_rot, "predict.rot_g", (3,)).expand(*bs, 3).contiguous()
    pred_shift = check_f32(pred_shift, "predict.shift_g", (3,)).expand(*bs, 3).contiguous()
    t = t.to(device=dev, dtype=torch.int64)
    if t.numel() == 1:
        t, t_stride = t.reshape(1).contiguous(), 0
    else:
        t, t_stride = _rows_t(t, bs, dev), 1
    recip, recipm1 = check_f32(recip, "sqrt_recip_alphas_cumprod"), check_f32(recipm1, "sqrt_recipm1_alphas_cumprod")
    coef1, coef2 = check_f32(coef1, "posterior_mean_coef1"), check_f32(coef2, "posterior_mean_coef2")
    sigma = check_f32(sigma, "sigma")
    T = recip.numel()
    trap_loc = None
    if post_cdf is not None:
        post_cdf = check_f32(post_cdf, "post_cdf", (CDF_POINTS,))
        if post_cdf.numel() != T * CDF_POINTS:
            raise ValueError("posterior cdf table must have one row per timestep")
        _check_guide(post_guide, T, "post_guide")
        _, _, trap_loc = cdf_grid(dev)
    seed_dev = _seed_tensor(seed, dev)
    if seed_dev is not None:
        if post_cdf is None or t_stride != 0 or rng_offset is None:
            raise ValueError("a device seed needs a shared step index, post_cdf and an explicit rng_offset")
    elif post_cdf is not None and (seed is None or rng_offset is None):
        seed, rng_offset = rng.next()
    rot_out, shift_out = torch.empty_like(rot_t), torch.empty_like(shift_t)
    if seed_dev is not None:  # CUDA-graph replayable step: the seed is read on the device when the kernel runs
        call("so3d_se3_p_sample_dseed_f32", ptr(rot_t), ptr(shift_t), ptr(pred_rot), ptr(pred_shift), ptr(t), ptr(recip), ptr(recipm1), ptr(coef1),
             ptr(coef2), ptr(sigma), T, ptr(post_cdf), ptr(trap_loc), float(shift_scale), ptr(seed_dev), int(rng_offset), int(row_offset),
             ptr(rot_out), ptr(shift_out), n, device=dev)
        return rot_out, shift_out
    call("so3d_se3_p_sample_f32", ptr(rot_t), ptr(shift_t), ptr(pred_rot), ptr(pred_shift), ptr(t), t_stride, ptr(recip), ptr(recipm1),
         ptr(coef1), ptr(coef2), ptr(sigma), T, ptr(post_cdf), ptr(post_guide), ptr(trap_loc), float(shift_scale), seed or 0, rng_offset or 0,
         int(row_offset), ptr(rot_out), ptr(shift_out), n, device=dev)
    return rot_out, shift_out


# ---------------------------------------------------------------------------------------------
# data side: Bingham quaternions (distributions.py:113-127), optionally straight to rotation matrices
# ---------------------------------------------------------------------------------------------
def bingham_sample(scale_tril, shape, z=None, seed=None, rng_offset=None, row_offset=0, want_quat=True, want_rmat=False):
    """scale_tril (4,4) CUDA float32 -> unit quaternions (*shape,4) and/or rotation matrices (*shape,3,3) in ONE
    launch.  z: optional explicit standard normals (*shape,4)."""
    scale_tril = check_f32(scale_tril, "scale_tril", (4, 4))
    if scale_tril.numel() != 16:
        raise ValueError("the fused Bingham sampler takes a single (4,4) scale_tril (no batch of covariances)")
    dev = scale_tril.device
    shape = tuple(int(d) for d in shape)
    n = 1
    for d in shape:
        n *= d
    if z is not None:
        z = check_f32(z, "z", (4,)).expand(*shape, 4).contiguous()
    if seed is None or rng_offset is None:
        seed, rng_offset = rng.next()
    if not (want_quat or want_rmat):
        raise ValueError("nothing to compute")
    q = torch.empty(*shape, 4, dtype=torch.float32, device=dev) if want_quat else None
    R = torch.empty(*shape, 3, 3, dtype=torch.float32, device=dev) if want_rmat else None
    call("so3d_bingham_sample_f32", ptr(scale_tril), ptr(z), seed, rng_offset, int(row_offset), ptr(q), ptr(R), n, device=dev)
    if want_quat and want_rmat:
        return q, R
    return q if want_quat else R


# ---------------------------------------------------------------------------------------------
# evaluation: all-pairs kernel sums (util.py:254-285 MMD)
# ---------------------------------------------------------------------------------------------
PAIR_KERNELS = {"gaussian": _lib.PAIR_GAUSSIAN, "cosine": _lib.PAIR_COSINE}
_pair_ws = {}


def pair_kernel_sums(X, Y=None, kernel="gaussian", shard=0, nshards=1):
    """X (nx,3,3), Y (ny,3,3) or None -> float64 (3,) = [sum_ij k(X_i,X_j), sum_ij k(Y_i,Y_j), sum_ij k(X_i,Y_j)]
    in one fused launch (nothing of size nx*ny is materialised).  With nshards > 1 only this shard's share of the
    256x256 tile pairs is summed (add the results of all shards)."""
    X = check_f32(X, "X", (3, 3)).reshape(-1, 3, 3)
    dev = X.device
    Y = check_f32(Y, "Y", (3, 3)).reshape(-1, 3, 3) if Y is not None else None
    if kernel not in PAIR_KERNELS:
        raise ValueError(f"kernel must be one of {sorted(PAIR_KERNELS)}")
    key = str(dev)
    if key not in _pair_ws:
        sms = torch.cuda.get_device_properties(dev).multi_processor_count
        _pair_ws[key] = torch.empty(3 * 8 * sms, dtype=torch.float64, device=dev)
    ws = _pair_ws[key]
    out = torch.empty(3, dtype=torch.float64, device=dev)
    call("so3d_pair_kernel_sums_f32", ptr(X), X.shape[0], ptr(Y), 0 if Y is None else Y.shape[0], PAIR_KERNELS[kernel],
         int(shard), int(nshards), ptr(ws), ws.numel(), ptr(out), device=dev)
    return out


# ---------------------------------------------------------------------------------------------
# L2: fused diffusion steps
# ---------------------------------------------------------------------------------------------
def _seed_tensor(seed, dev):
    """A device-resident seed (one int64 element, its 64 bits are the Philox key) or None for a by-value seed."""
    if not isinstance(seed, torch.Tensor):
        return None
    if seed.device != dev or seed.dtype != torch.int64 or seed.numel() != 1 or not seed.is_contiguous():
        raise ValueError("a device seed must be a contiguous int64 tensor with one element on the data's device")
    return seed


def q_sample_fused(x0, t, sqrt_ac, sqrt_1m_ac, cdf, seed=None, rng_offset=None, row_offset=0,
                   want_target=True, want_noise=False, want_score=False, guide=None):
    """-> dict(x_t, target, noise, score) (absent entries are None)."""
    x0, bs, n = _rows9(x0, "x_start")
    dev = x0.device
    t = _rows_t(t, bs, dev)
    sqrt_ac = check_f32(sqrt_ac, "sqrt_alphas_cumprod")
    sqrt_1m_ac = check_f32(sqrt_1m_ac, "sqrt_one_minus_alphas_cumprod")
    cdf = check_f32(cdf, "cdf", (CDF_POINTS,))
    T = sqrt_ac.numel()
    if cdf.numel() != T * CDF_POINTS:
        raise ValueError("cdf table must have one row per timestep")
    _, _, trap_loc = cdf_grid(dev)
    seed_dev = _seed_tensor(seed, dev)
    if seed_dev is None and (seed is None or rng_offset is None):
        seed, rng_offset = rng.next()
    x_t = torch.empty_like(x0)
    target = torch.empty(*bs, 3, dtype=torch.float32, device=dev) if want_target else None
    if seed_dev is not None:  # CUDA-graph replayable launch: the seed is read on the device when the kernel runs
        if want_noise or want_score:
            raise ValueError("a device seed supports the x_t / target outputs only")
        _check_guide(guide, T, "guide")
        call("so3d_q_sample_dseed_f32", ptr(x0), ptr(t), ptr(sqrt_ac), ptr(sqrt_1m_ac), T, ptr(cdf), ptr(guide), ptr(trap_loc), ptr(seed_dev),
             int(rng_offset or 0), int(row_offset), ptr(x_t), ptr(target), n, device=dev)
        return {"x_t": x_t, "target": target, "noise": None, "score": None}
    noise = torch.empty_like(x0) if want_noise else None
    score = torch.empty(*bs, 3, dtype=torch.float32, device=dev) if want_score else None
    _check_guide(guide, T, "guide")
    call("so3d_q_sample_f32", ptr(x0), ptr(t), ptr(sqrt_ac), ptr(sqrt_1m_ac), T, ptr(cdf), ptr(guide), ptr(trap_loc), seed, rng_offset,
         int(row_offset), ptr(x_t), ptr(target), ptr(noise), ptr(score), n, device=dev)
    return {"x_t": x_t, "target": target, "noise": noise, "score": score}


def q_sample_given(x0, t, sqrt_ac, noise):
    x0, bs, n = _rows9(x0, "x_start")
    noise = check_f32(noise, "noise", (3, 3)).expand_as(x0).contiguous()
    t = _rows_t(t, bs, x0.device)
    sqrt_ac = check_f32(sqrt_ac, "sqrt_alphas_cumprod")
    out = torch.empty_like(x0)
    call("so3d_q_sample_given_f32", ptr(x0), ptr(t), ptr(sqrt_ac), sqrt_ac.numel(), ptr(noise), ptr(out), n, device=x0.device)
    return out


def p_sample_fused(x_t, pred, t, recip, recipm1, coef1, coef2, post_cdf=None, seed=None, rng_offset=None, row_offset=0,
                   want_x0_hat=False, post_guide=None):
    """Fused reverse step.  t: int64 tensor with one element (shared step) or one per row.
    post_cdf None -> posterior mean only.  -> out (...,3,3)[, x0_hat]"""
    x_t, bs, n = _rows9(x_t, "x")
    dev = x_t.device
    pred = check_f32(pred, "predict", (3,)).expand(*bs, 3).contiguous()
    t = t.to(device=dev, dtype=torch.int64)
    if t.numel() == 1:
        t, t_stride = t.reshape(1).contiguous(), 0
    else:
        t, t_stride = _rows_t(t, bs, dev), 1
    recip, recipm1 = check_f32(recip, "sqrt_recip_alphas_cumprod"), check_f32(recipm1, "sqrt_recipm1_alphas_cumprod")
    coef1, coef2 = check_f32(coef1, "posterior_mean_coef1"), check_f32(coef2, "posterior_mean_coef2")
    T = recip.numel()
    trap_loc = None
    if post_cdf is not None:
        post_cdf = check_f32(post_cdf, "post_cdf", (CDF_POINTS,))
        if post_cdf.numel() != T * CDF_POINTS:
            raise ValueError("posterior cdf table must have one row per timestep")
        _check_guide(post_guide, T, "post_guide")
        _, _, trap_loc = cdf_grid(dev)
        if not isinstance(seed, torch.Tensor) and (seed is None or rng_offset is None):
            seed, rng_offset = rng.next()
    out = torch.empty_like(x_t)
    x0_hat = torch.empty_like(x_t) if want_x0_hat else None
    seed_dev = _seed_tensor(seed, dev)
    if seed_dev is not None:  # CUDA-graph replayable step: the seed is read on the device when the kernel runs
        if post_cdf is None or t_stride != 0 or want_x0_hat or rng_offset is None:
            raise ValueError("a device seed needs a shared step index, post_cdf, an explicit rng_offset and no x0_hat output")
        call("so3d_p_sample_dseed_f32", ptr(x_t), ptr(pred), ptr(t), ptr(recip), ptr(recipm1), ptr(coef1), ptr(coef2), T, ptr(post_cdf),
             ptr(trap_loc), ptr(seed_dev), int(rng_offset), int(row_offset), ptr(out), n, device=dev)
        return out
    call("so3d_p_sample_f32", ptr(x_t), ptr(pred), ptr(t), t_stride, ptr(recip), ptr(recipm1), ptr(coef1), ptr(coef2), T,
         ptr(post_cdf), ptr(post_guide), ptr(trap_loc), seed or 0, rng_offset or 0, int(row_offset), ptr(out), ptr(x0_hat), n, device=dev)
    return (out, x0_hat) if want_x0_hat else out


def p_sample_loop_fused(x_t, pred, t_hi, t_lo, recip, recipm1, coef1, coef2, post_cdf, post_guide, seed=None, rng_offset=0, row_offset=0,
                        out=None):
    """The reverse steps t_hi .. t_lo in ONE launch (so3d_p_sample_loop_f32): `pred` is None (no denoiser: zero prediction)
    or a fixed (...,3) prediction per particle; step t draws its noise at rng_offset + t.  Bit-identical to calling
    p_sample_fused(x, pred, [t], ..., seed=seed, rng_offset=rng_offset + t) for t = t_hi .. t_lo.  -> x_{t_lo - 1}"""
    x_t, bs, n = _rows9(x_t, "x")
    dev = x_t.device
    if pred is not None:
        pred = check_f32(pred, "predict", (3,)).expand(*bs, 3).contiguous()
    recip, recipm1 = check_f32(recip, "sqrt_recip_alphas_cumprod"), check_f32(recipm1, "sqrt_recipm1_alphas_cumprod")
    coef1, coef2 = check_f32(coef1, "posterior_mean_coef1"), check_f32(coef2, "posterior_mean_coef2")
    T = recip.numel()
    post_cdf = check_f32(post_cdf, "post_cdf", (CDF_POINTS,))
    if post_cdf.numel() != T * CDF_POINTS:
        raise ValueError("posterior cdf table must have one row per timestep")
    if post_guide is None:
        raise ValueError("post_guide (ops.igso3_cdf_guide(post_cdf)) is required")
    _check_guide(post_guide, T, "post_guide")
    _, _, trap_loc = cdf_grid(dev)
    if seed is None:
        seed, base = rng.next()
        rng_offset = int(rng_offset) + (base << 20)   # a fresh block of step offsets per call
    if out is None:
        out = torch.empty_like(x_t)
    elif out.shape != x_t.shape or out.dtype != torch.float32 or out.device != dev or not out.is_contiguous():
        raise ValueError("out must be a contiguous float32 tensor shaped like x")
    call("so3d_p_sample_loop_f32", ptr(x_t), ptr(pred), int(t_hi), int(t_lo), ptr(recip), ptr(recipm1), ptr(coef1), ptr(coef2), T, ptr(post_cdf),
         ptr(post_guide), ptr(trap_loc), int(seed), int(rng_offset), int(row_offset), ptr(out), n, device=dev)
    return out


# ---------------------------------------------------------------------------------------------
# RotPredict denoiser fused with the reverse step (SURVEY 8f-4)
# ---------------------------------------------------------------------------------------------
ROTPREDICT_D = 65
ROTPREDICT_BLOB_FLOATS = 39424  # include/so3d.h SO3D_ROTPREDICT_BLOB_FLOATS


def rotpredict_pack(weights, biases):
    """Five nn.Linear weight / bias tensors (so3_train.py:26-36) -> packed tf32 hi/lo blob for the fused kernel."""
    if len(weights) != 5 or len(biases) != 5:
        raise ValueError("RotPredict has five Linear layers")
    ws = [check_f32(w.detach(), f"weight{i + 1}", (ROTPREDICT_D,)) for i, w in enumerate(weights)]
    bs = [check_f32(b.detach(), f"bias{i + 1}") for i, b in enumerate(biases)]
    shapes = [(ROTPREDICT_D, ROTPREDICT_D)] * 4 + [(3, ROTPREDICT_D)]
    for w, b, s in zip(ws, bs, shapes):
        if tuple(w.shape) != s or b.numel() != s[0]:
            raise ValueError(f"unexpected layer shape {tuple(w.shape)} / {tuple(b.shape)}; RotPredict(d_model=65, out_type='skewvec') expected")
    dev = ws[0].device
    blob = torch.empty(ROTPREDICT_BLOB_FLOATS, dtype=torch.float32, device=dev)
    args = []
    for w, b in zip(ws, bs):
        args += [ptr(w), ptr(b)]
    call("so3d_rotpredict_pack_f32", *args, ptr(blob), device=dev)
    return blob


def rotpredict_p_sample_fused(x_t, blob, c1_table, t, recip, recipm1, coef1, coef2, post_cdf=None, seed=None, rng_offset=None,
                              row_offset=0, want_out=True, want_pred=False):
    """Denoiser + reverse step in one launch.  t: int64 tensor with ONE element (step shared by the batch).
    post_cdf None -> posterior mean only.  -> out (...,3,3) and/or pred (...,3)"""
    x_t, bs, n = _rows9(x_t, "x")
    dev = x_t.device
    t = t.to(device=dev, dtype=torch.int64)
    if t.numel() != 1:
        raise ValueError("the fused denoiser step takes a step index shared by the batch (t.numel() == 1)")
    t = t.reshape(1).contiguous()
    blob = check_f32(blob, "blob")
    if blob.numel() != ROTPREDICT_BLOB_FLOATS:
        raise ValueError("blob must come from rotpredict_pack")
    recip, recipm1 = check_f32(recip, "sqrt_recip_alphas_cumprod"), check_f32(recipm1, "sqrt_recipm1_alphas_cumprod")
    coef1, coef2 = check_f32(coef1, "posterior_mean_coef1"), check_f32(coef2, "posterior_mean_coef2")
    T = recip.numel()
    c1_table = check_f32(c1_table, "c1_table", (ROTPREDICT_D,))
    if c1_table.numel() != T * ROTPREDICT_D:
        raise ValueError("c1_table must have one row per timestep")
    trap_loc = None
    if post_cdf is not None:
        post_cdf = check_f32(post_cdf, "post_cdf", (CDF_POINTS,))
        if post_cdf.numel() != T * CDF_POINTS:
            raise ValueError("posterior cdf table must have one row per timestep")
        _, _, trap_loc = cdf_grid(dev)
        if not isinstance(seed, torch.Tensor) and (seed is None or rng_offset is None):
            seed, rng_offset = rng.next()
    if not (want_out or want_pred):
        raise ValueError("nothing requested")
    out = torch.empty_like(x_t) if want_out else None
    pred = torch.empty(*bs, 3, dtype=torch.float32, device=dev) if want_pred else None
    seed_dev = _seed_tensor(seed, dev)
    if seed_dev is not None:
        if rng_offset is None:
            raise ValueError("a device seed needs an explicit rng_offset")
        call("so3d_rotpredict_p_sample_dseed_f32", ptr(x_t), ptr(blob), ptr(c1_table), ptr(t), ptr(recip), ptr(recipm1), ptr(coef1), ptr(coef2),
             T, ptr(post_cdf), ptr(trap_loc), ptr(seed_dev), int(rng_offset), int(row_offset), ptr(out), ptr(pred), n, device=dev)
        if want_out and want_pred:
            return out, pred
        return out if want_out else pred
    call("so3d_rotpredict_p_sample_f32", ptr(x_t), ptr(blob), ptr(c1_table), ptr(t), ptr(recip), ptr(recipm1), ptr(coef1), ptr(coef2), T,
         ptr(post_cdf), ptr(trap_loc), seed or 0, rng_offset or 0, int(row_offset), ptr(out), ptr(pred), n, device=dev)
    if want_out and want_pred:
        return out, pred
    return out if want_out else pred


def rotpredict_p_sample_loop(x_t, blob, c1_table, t_hi, t_lo, recip, recipm1, coef1, coef2, post_cdf, seed, row_offset=0):
    """The reverse steps t_hi .. t_lo (inclusive, descending) with the RotPredict denoiser in ONE launch; step t draws
    its noise at rng_offset = t.  seed: int (by value) or a device int64[1] tensor.  -> x_{t_lo - 1} (...,3,3)"""
    x_t, bs, n = _rows9(x_t, "x")
    dev = x_t.device
    blob = check_f32(blob, "blob")
    if blob.numel() != ROTPREDICT_BLOB_FLOATS:
        raise ValueError("blob must come from rotpredict_pack")
    recip, recipm1 = check_f32(recip, "sqrt_recip_alphas_cumprod"), check_f32(recipm1, "sqrt_recipm1_alphas_cumprod")
    coef1, coef2 = check_f32(coef1, "posterior_mean_coef1"), check_f32(coef2, "posterior_mean_coef2")
    T = recip.numel()
    c1_table = check_f32(c1_table, "c1_table", (ROTPREDICT_D,))
    post_cdf = check_f32(post_cdf, "post_cdf", (CDF_POINTS,))
    if c1_table.numel() != T * ROTPREDICT_D or post_cdf.numel() != T * CDF_POINTS:
        raise ValueError("c1_table and post_cdf must have one row per timestep")
    if not (0 <= int(t_lo) <= int(t_hi) < T):
        raise ValueError("need 0 <= t_lo <= t_hi < T")
    _, _, trap_loc = cdf_grid(dev)
    seed_dev = _seed_tensor(seed, dev)
    out = torch.empty_like(x_t)
    call("so3d_rotpredict_p_sample_loop_f32", ptr(x_t), ptr(blob), ptr(c1_table), int(t_hi), int(t_lo), ptr(recip), ptr(recipm1), ptr(coef1),
         ptr(coef2), T, ptr(post_cdf), ptr(trap_loc), 0 if seed_dev is not None else int(seed), ptr(seed_dev), int(row_offset), ptr(out), n, device=dev)
    return out
