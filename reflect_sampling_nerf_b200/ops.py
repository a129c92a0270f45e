"""Python-side operators over the C-ABI (one function / autograd.Function per kernel stage).

Tensors stay torch-owned; these wrappers only check shapes, allocate outputs and pass raw device
pointers + the current CUDA stream to `librsn_b200.so`.  No CPU path exists.

`count` arguments: an int32 device tensor [1] holding the number of valid rays of a bounce pass (ops.reflect_compact).
Buffers are then sized for the capacity (the row count of the inputs) and rows >= count are never read or written, so
the number of masked rays never has to visit the host (include/rsn_b200.h, `n_rays_dev`).
"""
from __future__ import annotations

import ctypes as _ct
import functools
from typing import Optional, Tuple

import torch
from torch import Tensor

from . import _lib

UNIFORM, RECIPROCAL = 0, 1
# bench.py sets PROFILE to a list to collect (kernel, start event, end event, algorithmic FLOPs, bytes) per launch of
# the instrumented kernels on the launching stream; None (default) = no events recorded.
PROFILE = None
FLOP_PER_POINT = {0: 1230592, 1: 1225472}   # SURVEY.md §8d (forward; primary figure used for every sample pass)
# algorithmic (FLOPs, HBM bytes) per point (field kernels) / per sample (K1, K2, K8) -- DESIGN.md §4, SURVEY.md §8d
KERNEL_WORK = {
    "field_fwd_kernel": (1230592, 68),
    "field_fwd_kernel[train]": (1230592, 68 + 32 + 37 * 128 + 288),      # 41 stash blocks, the 4 bottleneck ones not written
    "field_chain_kernel<normals>": (1019392, 288 + 4 * 128 + 12),
    "field_chain_kernel<backward>": (1179904, 288 + 35 * 128 + 160),         # 39 dY blocks, the 4 of dY_bott not written
    "field_chain_kernel<backward+area>": (1229056, 288 + 4 * 128 + 35 * 128 + 164),
    # every stash block that exists once: 37 activation + 35 dY blocks of 128 B per point (the 12 active jobs issue 82 block
    # reads per tile: 10 operands are read by two jobs)
    "field_wgrad_kernel": (1230592, 72 * 128),
    # K8 at C = 16 channels, per SAMPLE: sigma 4 + bin 4 + feat 64 in, weight 4 out | + dL/dw 4 in, dL/dsigma 4 + dL/dfeat 64 out
    "composite_fwd_kernel": (0, 76),
    "composite_bwd_kernel": (0, 144),
    # K1: 8 B out (+ 4 B jitter in) per bin; K2: weights 4 + bins 4 + jitter 4 in, 8 out per bin (SURVEY.md §8d: 16-20 B)
    "sample_spaced_kernel": (0, 12),
    "pdf_resample_kernel": (0, 20),
}


class _Prof:
    """CUDA-event bracket around one kernel launch on the launching stream, active only while PROFILE is a list.
    n_units = work units (points / samples / bins) at the launch capacity; with a device-side ray `count` the entry also
    carries (count tensor, rays at capacity) so that the reader can scale the work to the rays actually processed."""

    def __init__(self, name: str, n_units: int, count: Optional[Tensor] = None, cap_rays: int = 0):
        self.name, self.n, self.on = name, n_units, PROFILE is not None
        self.count, self.cap_rays = count, cap_rays

    def __enter__(self):
        if self.on:
            self.e0, self.e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            self.e0.record()
        return self

    def __exit__(self, *exc):
        if self.on and PROFILE is not None:
            self.e1.record()
            flop, nbytes = KERNEL_WORK[self.name]
            PROFILE.append((self.name, self.e0, self.e1, self.n * flop, self.n * nbytes, self.count, self.cap_rays))
        return False


# ----------------------------------------------------------------------------------------- the tape
# The training step's backward is a fixed sequence of ~20 kernel launches.  torch.autograd can run it (every stage below is an
# autograd.Function, which is what nerfstudio's Trainer uses through loss.backward()), but the engine hops threads and
# streams, which costs launch latency and cannot be captured in a CUDA graph on this PyTorch build.  TrainStep therefore
# records the SAME Function.forward / Function.backward static methods on this minimal tape (under torch.no_grad()) and
# replays them in reverse itself: one thread, one stream, nothing but the kernels.
class _Ctx:
    """What a Function's forward / backward touch on `ctx`."""

    def __init__(self, needs_input_grad) -> None:
        self.needs_input_grad, self.saved_tensors, self.nondiff = needs_input_grad, (), ()

    def save_for_backward(self, *tensors) -> None:
        self.saved_tensors = tensors

    def mark_non_differentiable(self, *tensors) -> None:
        self.nondiff = tuple(id(t) for t in tensors)

    def set_materialize_grads(self, value: bool) -> None:
        pass


class Tape:
    def __init__(self) -> None:
        self.records, self.live = [], set()

    def apply(self, fn, *args):
        ctx = _Ctx(tuple(isinstance(a, Tensor) and id(a) in self.live for a in args))
        outs = fn.forward(ctx, *args)
        outs_t = outs if isinstance(outs, tuple) else (outs,)
        for o in outs_t:
            if isinstance(o, Tensor) and id(o) not in ctx.nondiff:
                self.live.add(id(o))
        self.records.append((fn, ctx, args, outs_t))       # (holds the tensors: their ids stay unique)
        return outs

    def backward(self, root: Tensor, grad_root: Tensor) -> None:
        grads = {id(root): grad_root}
        for fn, ctx, args, outs in reversed(self.records):
            gouts = tuple(grads.pop(id(o), None) if isinstance(o, Tensor) else None for o in outs)
            if all(g is None for g in gouts) and not getattr(fn, "always_backward", False):
                continue
            gins = fn.backward(ctx, *gouts)
            gins = gins if isinstance(gins, tuple) else (gins,)
            for a, g in zip(args, gins):
                if g is None or not isinstance(a, Tensor):
                    continue
                prev = grads.get(id(a))
                grads[id(a)] = g if prev is None else prev + g
        self.records.clear()


TAPE: Optional[Tape] = None


def tape_apply(fn, *args):
    return fn.apply(*args) if TAPE is None else TAPE.apply(fn, *args)


def _f32c(t: Optional[Tensor]) -> Optional[Tensor]:
    if t is None:
        return None
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def _cnt(count: Optional[Tensor]):
    if count is None:
        return None
    if count.dtype != torch.int32 or not count.is_cuda:
        raise ValueError("count must be an int32 CUDA tensor")
    return count.data_ptr()


@functools.lru_cache(maxsize=32)
def _linspace_bins(n_samples: int, device: torch.device) -> Tensor:
    # table taken from torch itself so it is bit-identical to SpacedSampler's (SURVEY.md App. A.2)
    return torch.linspace(0.0, 1.0, n_samples + 1).to(device)


@functools.lru_cache(maxsize=32)
def _pdf_u_base(n_out: int, train: bool, device: torch.device) -> Tensor:
    nb = n_out + 1
    u = torch.linspace(0.0, 1.0 - (1.0 / nb), steps=nb)
    if not train:
        u = u + 1.0 / (2 * nb)
    return u.to(device)


# ----------------------------------------------------------------------------------------- K1
def sample_spaced(nears: Tensor, fars: Tensor, n_samples: int, kind: int, t_rand: Optional[Tensor] = None,
                  count: Optional[Tensor] = None, tan: float = 0.25) -> Tuple[Tensor, Tensor]:
    """-> (spacing bins [N,S+1], euclidean bins [N,S+1]).  t_rand: [N,S+1] or [N,1] in [0,1), None = eval."""
    nears, fars, t_rand = _f32c(nears.reshape(-1)), _f32c(fars.reshape(-1)), _f32c(t_rand)
    n = nears.shape[0]
    dev = nears.device
    spacing = torch.empty(n, n_samples + 1, device=dev, dtype=torch.float32)
    euclid = torch.empty_like(spacing)
    cols = 0 if t_rand is None else t_rand.shape[-1]
    if t_rand is not None and t_rand.shape[0] != n:
        raise ValueError(f"t_rand has {t_rand.shape[0]} rows for {n} rays")
    with _Prof("sample_spaced_kernel", n * (n_samples + 1), count, n):
        _lib.call("rsn_sample_spaced", _lib.ptr(nears), _lib.ptr(fars), _lib.ptr(_linspace_bins(n_samples, dev)),
                  _lib.ptr(t_rand), cols, kind, float(tan), _lib.ptr(spacing), _lib.ptr(euclid), n, n_samples, _cnt(count),
                  _lib.stream())
    return spacing, euclid


# ----------------------------------------------------------------------------------------- K2
def pdf_resample(weights: Tensor, spacing_bins: Tensor, nears: Tensor, fars: Tensor, n_out: int, kind: int,
                 rand: Optional[Tensor] = None, train: Optional[bool] = None, histogram_padding: float = 0.01,
                 return_inds: bool = False, count: Optional[Tensor] = None, tan: float = 0.25):
    """weights [N,S] (or [N,S,1]); spacing_bins [N,S+1] -> (spacing [N,n_out+1], euclid [N,n_out+1][, inds])."""
    if weights.dim() == 3:
        weights = weights[..., 0]
    weights, spacing_bins = _f32c(weights.detach()), _f32c(spacing_bins)
    nears, fars, rand = _f32c(nears.reshape(-1)), _f32c(fars.reshape(-1)), _f32c(rand)
    n, s = weights.shape
    if spacing_bins.shape != (n, s + 1):
        raise ValueError(f"spacing_bins must be [{n},{s + 1}], got {tuple(spacing_bins.shape)}")
    if train is None:
        train = rand is not None
    if train and rand is None:
        rand = torch.rand(n, n_out + 1, device=weights.device)
    if rand is not None and rand.shape != (n, n_out + 1):
        raise ValueError(f"rand must be [{n},{n_out + 1}], got {tuple(rand.shape)}")
    dev = weights.device
    out_s = torch.empty(n, n_out + 1, device=dev, dtype=torch.float32)
    out_e = torch.empty_like(out_s)
    inds = torch.empty(n, n_out + 1, device=dev, dtype=torch.int64) if return_inds else None
    with _Prof("pdf_resample_kernel", n * (n_out + 1), count, n):
        _lib.call("rsn_pdf_resample", _lib.ptr(weights), weights.stride(0), _lib.ptr(spacing_bins), _lib.ptr(nears),
                  _lib.ptr(fars), _lib.ptr(_pdf_u_base(n_out, bool(train), dev)), _lib.ptr(rand), kind, float(tan),
                  float(histogram_padding), _lib.ptr(out_s), _lib.ptr(out_e), _lib.ptr(inds), n, s, n_out,
                  _cnt(count), _lib.stream())
    return (out_s, out_e, inds) if return_inds else (out_s, out_e)


# ----------------------------------------------------------------------------------------- K8
_COMPOSITE_CHANNELS = (0, 1, 3, 4, 8, 16)


class _Composite(torch.autograd.Function):
    """sigma [N,S], bins [N,S+1] (euclidean, no grad), feat [N,S,C] or None
    -> weights [N,S], accumulation [N], median depth [N] (no grad), feat_out [N,C]."""

    @staticmethod
    def forward(ctx, sigma: Tensor, bins: Tensor, feat: Optional[Tensor], count: Optional[Tensor]):
        sigma, bins, feat = _f32c(sigma), _f32c(bins), _f32c(feat)
        n, s = sigma.shape
        c = 0 if feat is None else feat.shape[-1]
        if c not in _COMPOSITE_CHANNELS:
            raise ValueError(f"composite: channel count {c} not in {_COMPOSITE_CHANNELS}")
        if bins.shape != (n, s + 1):
            raise ValueError(f"composite: bins must be [{n},{s + 1}], got {tuple(bins.shape)}")
        dev = sigma.device
        weights = torch.empty(n, s, device=dev, dtype=torch.float32)
        acc = torch.empty(n, device=dev, dtype=torch.float32)
        depth = torch.empty(n, device=dev, dtype=torch.float32)
        feat_out = torch.empty(n, c, device=dev, dtype=torch.float32)
        with _Prof("composite_fwd_kernel", n * s if c == 16 else 0):
            _lib.call("rsn_composite_fwd", _lib.ptr(sigma), bins.data_ptr(), bins.data_ptr() + 4, s + 1,
                      _lib.ptr(feat), c, _lib.ptr(weights), _lib.ptr(acc), _lib.ptr(depth),
                      _lib.ptr(feat_out) if c else None, n, s, _cnt(count), _lib.stream())
        ctx.save_for_backward(sigma, bins, feat if feat is not None else sigma.new_empty(0))
        ctx.c, ctx.count = c, count
        ctx.mark_non_differentiable(depth)
        ctx.set_materialize_grads(False)
        return weights, acc, depth, feat_out

    @staticmethod
    def backward(ctx, g_w, g_acc, _g_depth, g_feat_out):
        sigma, bins, feat = ctx.saved_tensors
        c = ctx.c
        n, s = sigma.shape
        need_feat = c > 0 and ctx.needs_input_grad[2]
        g_sigma = torch.empty_like(sigma)
        g_feat = torch.empty_like(feat) if need_feat else None
        g_w, g_acc, g_feat_out = _f32c(g_w), _f32c(g_acc), _f32c(g_feat_out) if c else None
        with _Prof("composite_bwd_kernel", n * s if c == 16 else 0):
            _lib.call("rsn_composite_bwd", _lib.ptr(sigma), bins.data_ptr(), bins.data_ptr() + 4, s + 1,
                      _lib.ptr(feat) if c else None, c, _lib.ptr(g_w), _lib.ptr(g_acc), _lib.ptr(g_feat_out),
                      _lib.ptr(g_sigma), _lib.ptr(g_feat), n, s, _cnt(ctx.count), _lib.stream())
        return g_sigma, None, g_feat, None


class _Composite16(torch.autograd.Function):
    """The model's form: 16 feature channels, with optional riders on the same pass (include/rsn_b200.h):
    normals [N,S,3] (constant) -> the two per-ray normal-loss sums; blend -> clip(rgb + (1 - acc), 0, 1);
    detach_sigma -> no density gradient (bounce passes); count -> device-side ray count.
    -> weights [N,S], accumulation [N], median depth [N], feat_out [N,16], pred_normal_loss [N], orientation_loss [N],
       rgb_blend [N,3]   (the riders that were not asked for come back as empty tensors)"""

    @staticmethod
    def forward(ctx, sigma: Tensor, bins: Tensor, feat: Tensor, normals: Optional[Tensor], count: Optional[Tensor],
                blend: bool, detach_sigma: bool):
        sigma, bins, feat, normals = _f32c(sigma), _f32c(bins), _f32c(feat), _f32c(normals)
        n, s = sigma.shape
        if feat.shape != (n, s, 16) or bins.shape != (n, s + 1) or (normals is not None and normals.shape != (n, s, 3)):
            raise ValueError("composite16: expects sigma [N,S], bins [N,S+1], feat [N,S,16], normals [N,S,3]")
        dev = sigma.device
        weights = torch.empty(n, s, device=dev, dtype=torch.float32)
        acc, depth = (torch.empty(n, device=dev, dtype=torch.float32) for _ in range(2))
        pnl, ol = (torch.empty(n if normals is not None else 0, device=dev, dtype=torch.float32) for _ in range(2))
        feat_out = torch.empty(n, 16, device=dev, dtype=torch.float32)
        rgb = torch.empty(n if blend else 0, 3, device=dev, dtype=torch.float32)
        with _Prof("composite_fwd_kernel", n * s, count, n):
            _lib.call("rsn_composite16_fwd", _lib.ptr(sigma), bins.data_ptr(), bins.data_ptr() + 4, s + 1, _lib.ptr(feat),
                      _lib.ptr(normals), _lib.ptr(weights), _lib.ptr(acc), _lib.ptr(depth), _lib.ptr(feat_out),
                      _lib.ptr(pnl) if normals is not None else None, _lib.ptr(ol) if normals is not None else None,
                      _lib.ptr(rgb) if blend else None, n, s, _cnt(count), _lib.stream())
        ctx.save_for_backward(sigma, bins, feat, normals if normals is not None else sigma.new_empty(0), feat_out, acc)
        ctx.count, ctx.has_normals, ctx.blend, ctx.detach_sigma = count, normals is not None, blend, detach_sigma
        ctx.mark_non_differentiable(depth)
        ctx.set_materialize_grads(False)
        return weights, acc, depth, feat_out, pnl, ol, rgb

    @staticmethod
    def backward(ctx, g_w, g_acc, _g_depth, g_feat_out, g_pnl, g_ol, g_rgb):
        sigma, bins, feat, normals, feat_out, acc = ctx.saved_tensors
        n, s = sigma.shape
        want_sigma = ctx.needs_input_grad[0] and not ctx.detach_sigma
        g_sigma = torch.empty_like(sigma) if want_sigma else None
        g_feat = torch.empty_like(feat)
        # keep the contiguous copies alive until the launch is enqueued (a freed temporary's block is handed to the
        # next allocation at once)
        g_w, g_acc, g_feat_out, g_pnl, g_ol, g_rgb = (_f32c(t) for t in (g_w, g_acc, g_feat_out, g_pnl, g_ol, g_rgb))
        with _Prof("composite_bwd_kernel", n * s, ctx.count, n):
            _lib.call("rsn_composite16_bwd", _lib.ptr(sigma), bins.data_ptr(), bins.data_ptr() + 4, s + 1, _lib.ptr(feat),
                      _lib.ptr(normals) if ctx.has_normals else None, _lib.ptr(g_w), _lib.ptr(g_acc), _lib.ptr(g_feat_out),
                      _lib.ptr(g_pnl) if ctx.has_normals else None, _lib.ptr(g_ol) if ctx.has_normals else None,
                      _lib.ptr(g_rgb) if ctx.blend else None, _lib.ptr(feat_out), _lib.ptr(acc), _lib.ptr(g_sigma),
                      _lib.ptr(g_feat), n, s, _cnt(ctx.count), _lib.stream())
        return g_sigma, None, g_feat, None, None, None, None


def composite16(sigma: Tensor, bins: Tensor, feat: Tensor, normals: Optional[Tensor] = None,
                count: Optional[Tensor] = None, blend: bool = False, detach_sigma: bool = False):
    return tape_apply(_Composite16, sigma, bins, feat, normals, count, blend, detach_sigma)


def composite(sigma: Tensor, bins: Tensor, feat: Optional[Tensor] = None, count: Optional[Tensor] = None):
    """Alpha compositing of one ray batch (K8).  Returns (weights, accumulation, median_depth, feat_out)."""
    return tape_apply(_Composite, sigma, bins, feat, count)


def render_weights(weights: Tensor, feat: Optional[Tensor] = None, bins: Optional[Tensor] = None,
                   starts: Optional[Tensor] = None, ends: Optional[Tensor] = None):
    """The upstream renderers' call form: weights [N,S] (+ feat [N,S,C], C <= 16) -> accumulation [N], feat_out [N,C] or
    None, median depth [N] or None (needs bins [N,S+1] or starts/ends [N,S])."""
    weights, feat = _f32c(weights), _f32c(feat)
    n, s = weights.shape
    c = 0 if feat is None else feat.shape[-1]
    dev = weights.device
    acc = torch.empty(n, device=dev, dtype=torch.float32)
    feat_out = torch.empty(n, c, device=dev, dtype=torch.float32) if c else None
    depth, sp, ep, stride = None, None, None, 0
    if bins is not None:
        bins = _f32c(bins)
        sp, ep, stride = bins.data_ptr(), bins.data_ptr() + 4, s + 1
    elif starts is not None:
        starts, ends = _f32c(starts.reshape(n, s)), _f32c(ends.reshape(n, s))
        sp, ep, stride = starts.data_ptr(), ends.data_ptr(), s
    if sp is not None:
        depth = torch.empty(n, device=dev, dtype=torch.float32)
    _lib.call("rsn_render_weights", _lib.ptr(weights), _lib.ptr(feat), c, sp, ep, stride, _lib.ptr(acc), _lib.ptr(feat_out),
              _lib.ptr(depth), n, s, _lib.stream())
    return acc, feat_out, depth


def ipe_encode(x: Tensor, covs: Optional[Tensor] = None) -> Tensor:
    """NeRFEncoding(3, 16, 0, 16, include_input=True).forward(x, covs): [...,3], [...,3,3] -> [...,99] (csrc/encode.cu)."""
    xs, cv = _f32c(x.reshape(-1, 3)), None if covs is None else _f32c(covs.reshape(-1, 3, 3))
    out = torch.empty(xs.shape[0], 99, device=xs.device, dtype=torch.float32)
    _lib.call("rsn_ipe_encode", _lib.ptr(xs), _lib.ptr(cv), _lib.ptr(out), xs.shape[0], _lib.stream())
    return out.reshape(*x.shape[:-1], 99)


def ide_encode(directions: Tensor, roughness: Tensor) -> Tensor:
    """IntegratedSHEncoding.forward(directions, roughness): [...,3], [...,1] -> [...,34] (csrc/encode.cu)."""
    d, r = _f32c(directions.reshape(-1, 3)), _f32c(roughness.reshape(-1))
    if r.shape[0] != d.shape[0]:
        raise ValueError("ide_encode: one roughness per direction")
    out = torch.empty(d.shape[0], 34, device=d.device, dtype=torch.float32)
    _lib.call("rsn_ide_encode", _lib.ptr(d), _lib.ptr(r), _lib.ptr(out), d.shape[0], _lib.stream())
    return out.reshape(*directions.shape[:-1], 34)


# ----------------------------------------------------------------------------------------- K3+K4+K5+K7
MODE_SAMPLES, MODE_INF_COLOR = 0, 1
N_FEAT = 16
(F_RGB, F_DIFF, F_TINT, F_NORMAL, F_ROUGH_SIGMOID, F_NDOTD, F_RAW_DENSITY, F_ROUGH_SOFTPLUS) = (
    slice(0, 3), slice(3, 6), slice(6, 9), slice(9, 12), 12, 13, 14, 15)


def field_forward(wblob: Tensor, bias: Tensor, origins: Tensor, dirs: Tensor, pixel_area: Tensor,
                  bins: Tensor, count: Optional[Tensor] = None, want_aux: bool = False):
    """Fused field evaluation of every frustum sample of a ray batch (inference form, no autograd).
    origins/dirs [N,3], pixel_area [N] or [N,1], bins [N,S+1] euclidean -> sigma [N,S], feat [N,S,16][, aux [N,S,8]]."""
    origins, dirs, bins = _f32c(origins), _f32c(dirs), _f32c(bins)
    area = _f32c(pixel_area.reshape(-1))
    n, s = bins.shape[0], bins.shape[1] - 1
    if origins.shape != (n, 3) or dirs.shape != (n, 3) or area.shape[0] != n:
        raise ValueError("field_forward: origins/dirs must be [N,3] and pixel_area [N] for bins [N,S+1]")
    sigma = torch.empty(n, s, device=bins.device, dtype=torch.float32)
    feat = torch.empty(n, s, N_FEAT, device=bins.device, dtype=torch.float32)
    aux = torch.empty(n, s, 8, device=bins.device, dtype=torch.float32) if want_aux else None
    with _Prof("field_fwd_kernel", n * s, count, n):
        _lib.call("rsn_field_forward_train", _lib.ptr(wblob), _lib.ptr(bias), MODE_SAMPLES, _lib.ptr(origins),
                  _lib.ptr(dirs), _lib.ptr(area), _lib.ptr(bins), n, s, _lib.ptr(sigma), _lib.ptr(feat), None,
                  _lib.ptr(aux), _cnt(count), _lib.stream())
    return (sigma, feat, aux) if want_aux else (sigma, feat)


def field_inf_color(wblob: Tensor, bias: Tensor, dirs: Tensor, sqradius: Tensor, count: Optional[Tensor] = None) -> Tensor:
    """field.get_inf_color (field.py:190-201): dirs [M,3], sqradius [M] or [M,1] -> rgb [M,3]."""
    dirs, sq = _f32c(dirs), _f32c(sqradius.reshape(-1))
    m = dirs.shape[0]
    sigma = torch.empty(m, device=dirs.device, dtype=torch.float32)
    feat = torch.empty(m, N_FEAT, device=dirs.device, dtype=torch.float32)
    _lib.call("rsn_field_forward", _lib.ptr(wblob), _lib.ptr(bias), MODE_INF_COLOR, None, _lib.ptr(dirs),
              _lib.ptr(sq), None, m, 1, _lib.ptr(sigma), _lib.ptr(feat), _cnt(count), _lib.stream())
    return feat[:, :3]


def field_forward_points(wblob: Tensor, bias: Tensor, mean: Tensor, cov: Tensor, dirs: Tensor,
                         rho: Optional[Tensor] = None):
    """The network on caller-supplied Gaussians (the reference's method-level Field API): mean [P,3], cov [P,3,3],
    dirs [P,3], rho [P] or None -> sigma [P], feat [P,16], aux [P,8]."""
    mean, cov, dirs, rho = _f32c(mean), _f32c(cov), _f32c(dirs), _f32c(rho)
    p = mean.shape[0]
    if mean.shape != (p, 3) or cov.shape != (p, 3, 3) or dirs.shape != (p, 3) or (rho is not None and rho.numel() != p):
        raise ValueError("field_forward_points: expects mean [P,3], cov [P,3,3], dirs [P,3], rho [P]")
    sigma = torch.empty(p, device=mean.device, dtype=torch.float32)
    feat = torch.empty(p, N_FEAT, device=mean.device, dtype=torch.float32)
    aux = torch.empty(p, 8, device=mean.device, dtype=torch.float32)
    _lib.call("rsn_field_forward_points", _lib.ptr(wblob), _lib.ptr(bias), _lib.ptr(mean), _lib.ptr(cov), _lib.ptr(dirs),
              _lib.ptr(rho), p, _lib.ptr(sigma), _lib.ptr(feat), _lib.ptr(aux), _lib.stream())
    return sigma, feat, aux


def frustum_gaussians(origins: Tensor, dirs: Tensor, pixel_area: Tensor, bins: Tensor) -> Tuple[Tensor, Tensor]:
    """field.get_blob: -> mean [N,S,3], cov [N,S,3,3] (uncontracted)."""
    origins, dirs, bins, area = _f32c(origins), _f32c(dirs), _f32c(bins), _f32c(pixel_area.reshape(-1))
    n, s = bins.shape[0], bins.shape[1] - 1
    mean = torch.empty(n, s, 3, device=bins.device, dtype=torch.float32)
    cov = torch.empty(n, s, 3, 3, device=bins.device, dtype=torch.float32)
    _lib.call("rsn_frustum_gaussians", _lib.ptr(origins), _lib.ptr(dirs), _lib.ptr(area), _lib.ptr(bins), n, s,
              _lib.ptr(mean), _lib.ptr(cov), _lib.stream())
    return mean, cov


def contract(mean: Tensor, cov: Tensor) -> Tuple[Tensor, Tensor]:
    """field.contract: mean [...,3], cov [...,3,3] -> contracted mean, J cov J (diagonal ReLU'd)."""
    mean, cov = _f32c(mean), _f32c(cov)
    mo, co = torch.empty_like(mean), torch.empty_like(cov)
    _lib.call("rsn_contract", _lib.ptr(mean), _lib.ptr(cov), _lib.ptr(mo), _lib.ptr(co), mean.numel() // 3, _lib.stream())
    return mo, co


# ----------------------------------------------------------------------------------------- training kernels
@functools.lru_cache(maxsize=1)
def wgrad_layout():
    """(offsets [2*J], shapes [(rows, cols)]*J, total floats) of the rsn_field_wgrad gradient blob."""
    offs = (_ct.c_int64 * 64)()
    shp = (_ct.c_int64 * 64)()
    tot = _ct.c_int64(0)
    n = _lib.lib().rsn_field_wgrad_layout(offs, shp, _ct.byref(tot))
    return [int(offs[i]) for i in range(2 * n)], [(int(shp[2 * j]), int(shp[2 * j + 1])) for j in range(n)], int(tot.value)


def field_forward_train(wblob: Tensor, bias: Tensor, mode: int, origins: Optional[Tensor], dirs: Tensor,
                        area: Tensor, bins: Optional[Tensor], stash: Optional[Tensor] = None,
                        count: Optional[Tensor] = None):
    """Forward pass that also leaves the activation stash + aux for the backward kernels.
    mode 0: bins [N,S+1]; mode 1 (infinity colour): one point per ray.  -> sigma [N,S], feat [N,S,16], stash, aux"""
    dirs, area = _f32c(dirs), _f32c(area.reshape(-1))
    n = dirs.shape[0]
    if mode == MODE_SAMPLES:
        origins, bins = _f32c(origins), _f32c(bins)
        s = bins.shape[1] - 1
    else:
        s = 1
    dev = dirs.device
    sigma = torch.empty(n, s, device=dev, dtype=torch.float32)
    feat = torch.empty(n, s, N_FEAT, device=dev, dtype=torch.float32)
    aux = torch.empty(n, s, 8, device=dev, dtype=torch.float32)
    nbytes = _lib.lib().rsn_field_stash_bytes(n * s)
    if stash is None:
        stash = torch.empty(nbytes, device=dev, dtype=torch.uint8)
    elif stash.numel() < nbytes or stash.dtype != torch.uint8 or stash.device != dev:
        raise ValueError("field_forward_train: stash workspace too small")
    with _Prof("field_fwd_kernel[train]", n * s, count, n):
        _lib.call("rsn_field_forward_train", _lib.ptr(wblob), _lib.ptr(bias), mode, _lib.ptr(origins), _lib.ptr(dirs),
                  _lib.ptr(area), _lib.ptr(bins), n, s, _lib.ptr(sigma), _lib.ptr(feat), _lib.ptr(stash),
                  _lib.ptr(aux), _cnt(count), _lib.stream())
    return sigma, feat, stash, aux


def field_normals(wblob_t: Tensor, wd_bf16: Tensor, stash: Tensor, n: int, s: int) -> Tensor:
    """K6: -normalize(d raw_density / d contracted mean) of every sample of the pass that produced `stash`."""
    normals = torch.empty(n, s, 3, device=stash.device, dtype=torch.float32)
    with _Prof("field_chain_kernel<normals>", n * s):
        _lib.call("rsn_field_normals", _lib.ptr(wblob_t), _lib.ptr(wd_bf16), _lib.ptr(stash), n, s,
                  _lib.ptr(normals), _lib.stream())
    return normals


def field_backward(wblob_t: Tensor, stash: Tensor, mode: int, origins, dirs, area, bins, n: int, s: int,
                   g_sigma: Optional[Tensor], g_feat: Tensor, feat: Tensor, aux: Tensor, dy_stash: Tensor,
                   want_area: bool, count: Optional[Tensor] = None) -> Optional[Tensor]:
    """K5 dgrad chain: fills dy_stash; returns dL/d pixel_area (mode 0) / dL/d sqradius (mode 1) per POINT [n,s]
    when want_area."""
    g_area = torch.empty(n, s, device=stash.device, dtype=torch.float32) if want_area else None
    with _Prof("field_chain_kernel<backward+area>" if want_area else "field_chain_kernel<backward>", n * s, count, n):
        _lib.call("rsn_field_backward", _lib.ptr(wblob_t), _lib.ptr(stash), mode, _lib.ptr(origins), _lib.ptr(dirs),
                  _lib.ptr(area), _lib.ptr(bins), n, s, _lib.ptr(g_sigma), _lib.ptr(g_feat), _lib.ptr(feat),
                  _lib.ptr(aux), _lib.ptr(dy_stash), _lib.ptr(g_area), _cnt(count), _lib.stream())
    return g_area


def field_wgrad(stash: Tensor, dy_stash: Tensor, n_points: int, grad_blob: Tensor, count: Optional[Tensor] = None,
                points_per_ray: int = 1) -> None:
    """K5 wgrad: accumulates dW / db of every Linear over the pass into grad_blob (fp32, wgrad_layout()), in a fixed
    order (the same gradient every run).  The partial-sum workspace comes from the caching allocator, per call."""
    ws = torch.empty(_lib.lib().rsn_field_wgrad_workspace_bytes(), dtype=torch.uint8, device=grad_blob.device)
    with _Prof("field_wgrad_kernel", n_points, count, n_points // max(points_per_ray, 1)):
        _lib.call("rsn_field_wgrad", _lib.ptr(stash), _lib.ptr(dy_stash), n_points, _lib.ptr(grad_blob), _lib.ptr(ws),
                  _cnt(count), points_per_ray, _lib.stream())


def wgrad_finish(grad_blob: Tensor, w_bott: Tensor, b_bott: Tensor, w_mid: Tensor) -> None:
    """Once per step, after the last field_wgrad (and the all-reduce): derive the bottleneck layer's gradients and the
    bottleneck columns of d mlp_mid.layers.0.weight from G = dY_mid^T h7 = rows 64-191 of wgrad job 10
    (include/rsn_b200.h: rsn_field_wgrad_finish).
    CPU tensors (the gloo test of the flush path) take the same algebra through torch."""
    if grad_blob.is_cuda:
        _lib.call("rsn_field_wgrad_finish", _lib.ptr(grad_blob), _lib.ptr(_f32c(w_bott.detach())),
                  _lib.ptr(_f32c(b_bott.detach())), _lib.ptr(_f32c(w_mid.detach())), _lib.stream())
        return
    offs, shapes, _ = wgrad_layout()
    g = grad_blob[offs[20] + 64 * 256: offs[20] + 192 * 256].view(128, 256)      # rows 64-191 of job 10's region
    db_mid = grad_blob[offs[21] + 64: offs[21] + 192]
    w_mb = w_mid.detach()[:, 34:]
    grad_blob[offs[18]: offs[18] + 256 * 256] = (w_mb.T @ g).reshape(-1)
    grad_blob[offs[19]: offs[19] + 256] = w_mb.T @ db_mid
    grad_blob[offs[24]: offs[24] + 128 * 256] = (g @ w_bott.detach().T + torch.outer(db_mid, b_bott.detach())).reshape(-1)
    grad_blob[offs[25]: offs[25] + 128] = db_mid


PACK_ORDER = ([f"mlp_base.layers.{l}.weight" for l in range(8)] + [f"mlp_base.layers.{l}.bias" for l in range(8)]
              + [f"{m}.{k}" for m in ("field_output_bottleneck.net", "mlp_mid.layers.0", "field_output_mid.net",
                                      "field_output_density.net", "field_output_normals.net",
                                      "field_output_roughness.net", "field_output_diff.net", "field_output_tint.net")
                 for k in ("weight", "bias")])


def pack_field(named_params, out=None) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """One-launch packing of the field's fp32 parameters (dict name -> CUDA tensor) into
    (forward blob, bias vector, transposed blob, bf16 density row) -- csrc/pack.cu.  `out` = the four tensors of an
    earlier call to overwrite in place (static addresses: CUDA graphs)."""
    tensors = [_f32c(named_params[k].detach()) for k in PACK_ORDER]
    dev = tensors[0].device
    ptrs = (_ct.c_void_p * len(tensors))(*[_lib.ptr(t) for t in tensors])
    if out is not None:
        wblob, bias, wblob_t, wd = out
    else:
        wblob = torch.empty(_lib.lib().rsn_field_blob_bytes(), dtype=torch.uint8, device=dev)
        wblob_t = torch.empty(_lib.lib().rsn_field_blob_t_bytes(), dtype=torch.uint8, device=dev)
        bias = torch.empty(_lib.lib().rsn_field_bias_count(), dtype=torch.float32, device=dev)
        wd = torch.empty(256, dtype=torch.bfloat16, device=dev)
    _lib.call("rsn_pack_field", ptrs, _lib.ptr(wblob), _lib.ptr(wblob_t), _lib.ptr(bias), _lib.ptr(wd), _lib.stream())
    return wblob, bias, wblob_t, wd


@functools.lru_cache(maxsize=1)
def flat_layout():
    """(offsets of the 32 parameters of PACK_ORDER in the flat gradient vector, total length)."""
    offs = (_ct.c_int64 * 32)()
    total = _lib.lib().rsn_field_flat_layout(offs)
    return [int(o) for o in offs], int(total)


def unpack_grads_flat(grad_blob: Tensor, flat: Tensor) -> Tensor:
    """Gradient blob of field_wgrad -> flat fp32 gradient vector (one launch, csrc/pack.cu)."""
    _lib.call("rsn_unpack_grads", _lib.ptr(grad_blob), _lib.ptr(flat), _lib.stream())
    return flat


def radam_step(named_params, flat_grad: Tensor, exp_avg: Tensor, exp_avg_sq: Tensor, step: Tensor, counter: Tensor,
               lr_out: Optional[Tensor], lr: float, lr_final: float = 0.0, max_steps: int = 0,
               betas=(0.9, 0.999), eps: float = 1e-15, grad_scale: float = 1.0) -> None:
    """Fused RAdam (+ exponential lr decay) over the 32 trained parameters (csrc/optim.cu); `step` int64 [1] and
    `counter` int32 [1] live on the device."""
    tensors = [named_params[k] for k in PACK_ORDER]
    for t in tensors:
        if t.dtype != torch.float32 or not t.is_contiguous():
            raise ValueError("radam_step: parameters must be contiguous fp32")
    ptrs = (_ct.c_void_p * len(tensors))(*[_lib.ptr(t) for t in tensors])
    _lib.call("rsn_radam_step", ptrs, _lib.ptr(flat_grad), _lib.ptr(exp_avg), _lib.ptr(exp_avg_sq), _lib.ptr(step),
              _lib.ptr(counter), _lib.ptr(lr_out), float(lr), float(lr_final), int(max_steps), float(betas[0]),
              float(betas[1]), float(eps), float(grad_scale), _lib.stream())


# ----------------------------------------------------------------------------------------- K9
def reflect_setup(comp16: Tensor, acc: Tensor, depth: Tensor, origins: Tensor, dirs: Tensor, clamp01: bool):
    """Per-ray quantities of the bounce from the composited fine pass (model.py:215-229,267-271), all detached:
    -> diff [N,3], tint [N,3], normal [N,3], n_dot_d [N,1], mask [N] uint8, bounce origins [N,3], bounce dirs [N,3]."""
    comp16, acc, depth = _f32c(comp16.detach()), _f32c(acc.detach().reshape(-1)), _f32c(depth.detach().reshape(-1))
    origins, dirs = _f32c(origins), _f32c(dirs)
    n, dev = comp16.shape[0], comp16.device
    diff, tint, nrm, o2, wr = (torch.empty(n, 3, device=dev, dtype=torch.float32) for _ in range(5))
    ndd = torch.empty(n, 1, device=dev, dtype=torch.float32)
    mask = torch.empty(n, device=dev, dtype=torch.uint8)
    _lib.call("rsn_reflect_setup", _lib.ptr(comp16), _lib.ptr(acc), _lib.ptr(depth), _lib.ptr(origins), _lib.ptr(dirs),
              int(clamp01), _lib.ptr(diff), _lib.ptr(tint), _lib.ptr(nrm), _lib.ptr(ndd), _lib.ptr(mask), _lib.ptr(o2),
              _lib.ptr(wr), n, _lib.stream())
    return diff, tint, nrm, ndd, mask, o2, wr


def reflect_compact(mask: Tensor):
    """Device-side `x[mask]` bookkeeping: mask [N] uint8/bool -> idx [N] int64 (first `count` entries = ascending indices
    of the masked rays), inv [N] int32 (rank of a ray among the masked rays or -1), count [1] int32.  No host sync."""
    if mask.dtype == torch.bool:
        mask = mask.view(torch.uint8)
    mask = mask.contiguous()
    n, dev = mask.shape[0], mask.device
    idx = torch.empty(n, device=dev, dtype=torch.int64)
    inv = torch.empty(n, device=dev, dtype=torch.int32)
    count = torch.empty(1, device=dev, dtype=torch.int32)
    _lib.call("rsn_reflect_compact", _lib.ptr(mask), _lib.ptr(idx), _lib.ptr(inv), _lib.ptr(count), n, _lib.stream())
    return idx, inv, count


class _ReflectBundle(torch.autograd.Function):
    """Reflected RayBundle of the masked rays (model.py:267-289): rows j < count = ray idx[j].
    -> origins [N,3], dirs [N,3] (detached), sqradius [N], pixel_area [N] (grad -> roughness = comp16[:, 12])."""

    @staticmethod
    def forward(ctx, comp16: Tensor, idx: Tensor, inv: Tensor, count: Tensor, o2_all: Tensor, wr_all: Tensor, ndd: Tensor):
        comp16 = _f32c(comp16)
        n, dev = comp16.shape[0], comp16.device
        o2, wr = (torch.empty(n, 3, device=dev, dtype=torch.float32) for _ in range(2))
        sqr, area = (torch.empty(n, device=dev, dtype=torch.float32) for _ in range(2))
        _lib.call("rsn_reflect_bundle_fwd", _lib.ptr(idx), _lib.ptr(count), _lib.ptr(o2_all), _lib.ptr(wr_all), _lib.ptr(ndd),
                  _lib.ptr(comp16), _lib.ptr(o2), _lib.ptr(wr), _lib.ptr(sqr), _lib.ptr(area), n, _lib.stream())
        ctx.save_for_backward(comp16, inv, ndd)
        ctx.mark_non_differentiable(o2, wr)
        ctx.set_materialize_grads(False)
        return o2, wr, sqr, area

    @staticmethod
    def backward(ctx, _g_o2, _g_wr, g_sqr, g_area):
        comp16, inv, ndd = ctx.saved_tensors
        if g_sqr is None and g_area is None:
            return (None,) * 7
        g_sqr, g_area = _f32c(g_sqr), _f32c(g_area)
        g_comp = torch.empty_like(comp16)
        _lib.call("rsn_reflect_bundle_bwd", _lib.ptr(inv), _lib.ptr(ndd), _lib.ptr(comp16), _lib.ptr(g_sqr), _lib.ptr(g_area),
                  _lib.ptr(g_comp), comp16.shape[0], _lib.stream())
        return g_comp, None, None, None, None, None, None


def reflect_bundle(comp16, idx, inv, count, o2_all, wr_all, ndd):
    return tape_apply(_ReflectBundle, comp16, idx, inv, count, o2_all, wr_all, _f32c(ndd.reshape(-1)))


class _ReflectCompose(torch.autograd.Function):
    """out[r] = 1 - acc_fine[r] (white background rest, gradient to acc_fine: App. B Q10) for rays that do not bounce, else
    clip(diff[r] + tint[r] * (comp16[j, :3] + bg[j] * (1 - acc_r[j])), 0, 1), j = inv[r]   (model.py:240-241,311-313).
    depth_r [cap] (optional) is scattered to [N] (0 where no bounce).  -> out [N,3], depth_out [N] (or empty)"""

    @staticmethod
    def forward(ctx, acc_fine, diff, tint, inv, comp16, bg, acc_r, depth_r, clamp_inner: bool):
        acc_fine, diff, tint, comp16, bg, acc_r, depth_r = (
            _f32c(t) for t in (acc_fine.reshape(-1), diff, tint, comp16, bg, acc_r.reshape(-1),
                               None if depth_r is None else depth_r.reshape(-1)))
        n = acc_fine.shape[0]
        out = torch.empty(n, 3, device=acc_fine.device, dtype=torch.float32)
        depth_out = torch.empty(n if depth_r is not None else 0, device=acc_fine.device, dtype=torch.float32)
        _lib.call("rsn_reflect_compose_fwd", _lib.ptr(acc_fine), _lib.ptr(diff), _lib.ptr(tint), _lib.ptr(inv), _lib.ptr(comp16),
                  comp16.shape[1], _lib.ptr(bg), _lib.ptr(acc_r), int(clamp_inner), _lib.ptr(out), _lib.ptr(depth_r),
                  _lib.ptr(depth_out) if depth_r is not None else None, n, _lib.stream())
        ctx.save_for_backward(diff, tint, inv, comp16, bg, acc_r)
        ctx.acc_shape = None
        ctx.mark_non_differentiable(depth_out)
        ctx.set_materialize_grads(False)
        return out, depth_out

    @staticmethod
    def backward(ctx, g_out, _g_depth):
        diff, tint, inv, comp16, bg, acc_r = ctx.saved_tensors
        if g_out is None:
            return (None,) * 9
        g_out = _f32c(g_out)
        n = g_out.shape[0]
        g_comp = torch.empty_like(comp16)
        g_bg = torch.empty_like(bg)
        g_acc = torch.empty(n, device=g_out.device, dtype=torch.float32)
        _lib.call("rsn_reflect_compose_bwd", _lib.ptr(g_out), _lib.ptr(diff), _lib.ptr(tint), _lib.ptr(inv), _lib.ptr(comp16),
                  comp16.shape[1], _lib.ptr(bg), _lib.ptr(acc_r), _lib.ptr(g_comp), _lib.ptr(g_bg), _lib.ptr(g_acc), n,
                  _lib.stream())
        return g_acc, None, None, None, g_comp, g_bg, None, None, None


def reflect_compose(acc_fine, diff, tint, inv, comp16, bg, acc_r, depth_r=None, clamp_inner: bool = False):
    """-> (out [N,3], depth_out [N] or empty).  acc_fine [N] (or [N,1]) carries the gradient of the fallback rows."""
    if comp16.shape[1] != 16:
        raise ValueError("reflect_compose: comp16 must be the composited 16-channel feature rows")
    return tape_apply(_ReflectCompose, acc_fine, diff, tint, inv, comp16, bg, acc_r, depth_r, clamp_inner)


# ----------------------------------------------------------------------------------------- losses
LOSS_KEYS = ("loss_mid_coarse", "loss_mid_fine", "loss_reflect_mid_coarse", "loss_reflect_mid_fine",
             "predicted_normal_loss_coarse", "predicted_normal_loss_fine", "orientation_loss_coarse",
             "orientation_loss_fine")


class _FusedLoss(torch.autograd.Function):
    """get_loss_dict (model.py:395-429) in one launch: -> terms [8] (scaled, LOSS_KEYS order), total []."""

    @staticmethod
    def forward(ctx, rgb_c, rgb_f, refl_c, refl_f, image, pnl_c, pnl_f, ol_c, ol_f, coef, workspace):
        preds = [_f32c(t) for t in (rgb_c, rgb_f, refl_c, refl_f)]
        image = _f32c(image)
        sums = [_f32c(t) if t is not None else None for t in (pnl_c, pnl_f, ol_c, ol_f)]
        n = image.shape[0]
        out = torch.empty(9, device=image.device, dtype=torch.float32)
        _lib.call("rsn_loss_fwd", *[_lib.ptr(t) for t in preds], _lib.ptr(image), *[_lib.ptr(t) for t in sums],
                  _lib.ptr(coef), _lib.ptr(out), _lib.ptr(workspace), n, _lib.stream())
        ctx.save_for_backward(*preds, image, coef)
        ctx.have_sums = [t is not None for t in sums]
        ctx.set_materialize_grads(False)
        return out[:8], out[8]

    @staticmethod
    def backward(ctx, g_terms, g_total):
        *preds, image, coef = ctx.saved_tensors
        n = image.shape[0]
        g_terms, g_total = _f32c(g_terms), _f32c(g_total)
        g_pred = [torch.empty_like(p) for p in preds]
        g_sums = [torch.empty(n, device=image.device, dtype=torch.float32) if h else None for h in ctx.have_sums]
        _lib.call("rsn_loss_bwd", *[_lib.ptr(t) for t in preds], _lib.ptr(image), _lib.ptr(coef), _lib.ptr(g_terms),
                  _lib.ptr(g_total), *[_lib.ptr(t) for t in g_pred], *[_lib.ptr(t) for t in g_sums], n, _lib.stream())
        return (*g_pred, None, *g_sums, None, None)


def loss_workspace(device) -> Tensor:
    return torch.zeros(_lib.lib().rsn_loss_workspace_bytes(), dtype=torch.uint8, device=device)


def fused_loss(rgb_c, rgb_f, refl_c, refl_f, image, pnl_c, pnl_f, ol_c, ol_f, coef: Tensor, workspace: Tensor):
    return tape_apply(_FusedLoss, rgb_c, rgb_f, refl_c, refl_f, image, pnl_c, pnl_f, ol_c, ol_f, coef, workspace)


class _InfColorRGB(torch.autograd.Function):
    """bg = feat[:, 0, 0:3] of the infinity-colour pass ([M,1,16] -> [M,3], contiguous) and its scatter-back."""

    @staticmethod
    def forward(ctx, feat: Tensor):
        ctx.shape = feat.shape
        return feat[:, 0, 0:3].contiguous()

    @staticmethod
    def backward(ctx, g):
        if g is None:
            return None
        gf = g.new_zeros(ctx.shape)
        gf[:, 0, 0:3] = g
        return gf


def inf_color_rgb(feat_bg: Tensor) -> Tensor:
    return tape_apply(_InfColorRGB, feat_bg)


# ----------------------------------------------------------------------------------------- f1: ray generation
def raygen(c2w: Tensor, intrinsics: Tensor, height: int, width: int, n_rays: int, rand: Optional[Tensor] = None,
           pixels: Optional[Tensor] = None, images: Optional[Tensor] = None):
    """Pixel sampling + camera rays + target gather (csrc/raygen.cu).  c2w [V,3,4], intrinsics [V,4] = fx, fy, cx, cy;
    rand [N,3] uniform or pixels [N,3] int64 (cam, y, x); images [V,H,W,C] uint8 or None.
    -> origins [N,3], dirs [N,3], pixel_area [N,1], pixels [N,3] int64, target [N,3] or None"""
    c2w, intrinsics, rand = _f32c(c2w), _f32c(intrinsics), _f32c(rand)
    dev, v = c2w.device, c2w.shape[0]
    if (rand is None) == (pixels is None):
        raise ValueError("raygen: exactly one of rand / pixels")
    if images is not None and (images.dtype != torch.uint8 or images.shape[:3] != (v, height, width)):
        raise ValueError("raygen: images must be uint8 [V,H,W,C]")
    o, d = (torch.empty(n_rays, 3, device=dev, dtype=torch.float32) for _ in range(2))
    area = torch.empty(n_rays, 1, device=dev, dtype=torch.float32)
    pix = torch.empty(n_rays, 3, device=dev, dtype=torch.int64)
    target = torch.empty(n_rays, 3, device=dev, dtype=torch.float32) if images is not None else None
    images = images.contiguous() if images is not None else None
    pixels = pixels.contiguous() if pixels is not None else None
    _lib.call("rsn_raygen", _lib.ptr(c2w), _lib.ptr(intrinsics), _lib.ptr(rand), _lib.ptr(pixels), _lib.ptr(images),
              images.shape[-1] if images is not None else 0, v, height, width, _lib.ptr(o), _lib.ptr(d), _lib.ptr(area),
              _lib.ptr(pix), _lib.ptr(target), n_rays, _lib.stream())
    return o, d, area, pix, target
