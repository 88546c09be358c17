"""Temporal up-sampling of joint trajectories to the radar sampling rate on the GPU -- the B200
replacement for the reference data loader's `Dataset.pad_frames` (utils.py:134-140) plus the float32
cast of `Dataset.__getitem__` (utils.py:128-132): Gaussian smoothing along time (scipy
`gaussian_filter1d`, reflect boundary, float64 accumulation, float32 result) followed by not-a-knot
cubic interpolation (scipy `interp1d(..., 'cubic')`) to `num_pad_frames * T` frames, evaluated in
float64 and rounded to float32.  One CUDA kernel through the C ABI (`vr_pad_frames_f32`); no CPU path.
Differentiable: under grad mode, an `x` that requires grad gets dL/dx from `vr_pad_frames_backward_f32` (the transpose
of the float64 linear operator; the float32 roundings pass the gradient through as a dtype cast does)."""
import ctypes

import torch

from . import _cabi


def _launch(xb, k, sigma, out):
    N, _, T, V, M = xb.shape
    with torch.cuda.device(xb.device):
        stream = torch.cuda.current_stream(xb.device).cuda_stream
        rc = _cabi.lib().vr_pad_frames_f32(xb.data_ptr(), N, T, V, M, k, ctypes.c_float(float(sigma)),
                                           out.data_ptr(), ctypes.c_void_p(stream))
    _cabi.check(rc)


class _PadFramesFunction(torch.autograd.Function):
    """pad_frames with a backward pass (C ABI vr_pad_frames_backward_f32).  `out` is written in place and marked dirty,
    so that the `out=` form carries the graph too."""

    @staticmethod
    def forward(ctx, xb, k, sigma, out):
        _launch(xb, k, sigma, out)
        ctx.mark_dirty(out)
        ctx.dims = (tuple(xb.shape), k, sigma)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        (N, C, T, V, M), k, sigma = ctx.dims
        g = grad_out.contiguous().to(torch.float32)
        gx = torch.empty((N, C, T, V, M), dtype=torch.float32, device=g.device)
        with torch.cuda.device(g.device):
            stream = torch.cuda.current_stream(g.device).cuda_stream
            rc = _cabi.lib().vr_pad_frames_backward_f32(g.data_ptr(), N, T, V, M, k, ctypes.c_float(float(sigma)),
                                                        gx.data_ptr(), ctypes.c_void_p(stream))
        _cabi.check(rc)
        return gx, None, None, None


def pad_frames(x, num_pad_frames=250, sigma=3, out=None):
    """x: (N,3,T,V,M) or a single sample (3,T,V,M), float32 CUDA tensor -> same rank with
    `num_pad_frames * T` frames.  Defaults are the reference's (utils.py:105).  Differentiable with
    respect to x (also through `out=`); without grad the result carries no graph."""
    if not isinstance(x, torch.Tensor) or x.dim() not in (4, 5):
        raise ValueError("expected a (N,3,T,V,M) or (3,T,V,M) tensor")
    if x.dtype != torch.float32:
        raise ValueError("pad_frames takes float32 (the dataset's dtype, utils.py:124); got %s" % x.dtype)
    if not x.is_cuda:
        raise RuntimeError("pad_frames (B200) has no CPU path: move x to a CUDA device")
    single = x.dim() == 4
    xb = (x.unsqueeze(0) if single else x).contiguous()
    N, C, T, V, M = xb.shape
    k = int(num_pad_frames)
    shape = (N, C, k * T, V, M)
    if out is None:
        out = torch.empty(shape, dtype=torch.float32, device=x.device)
    elif tuple(out.shape) != shape or out.dtype != torch.float32 or not out.is_contiguous() or out.device != x.device:
        raise ValueError("out must be a contiguous float32 tensor of shape %s on %s" % (shape, x.device))
    if C != 3:
        raise ValueError("expected 3 coordinate planes, got %d" % C)
    if N == 0:
        return out[0] if single else out
    if torch.is_grad_enabled() and x.requires_grad:
        out = _PadFramesFunction.apply(xb, k, sigma, out)
    else:
        _launch(xb, k, sigma, out)
    return out[0] if single else out


def pad_frames_notebook(data, num_pad_frames=1, sigma=3, planar=False):
    """The notebook's `utils.pad_frames` (reference utils.py:82-89) on the device: `data` is one body's (T, V, C) array --
    or a batch (N, T, V, C) -- float64 or float32 CUDA tensor; Gaussian smoothing along the JOINT axis (the reference's
    quirk, kept), not-a-knot cubic interpolation in time to `num_pad_frames * T` frames in float64, float32 result (the
    cast of `torch.Tensor(...)` in virtual_radar_example.ipynb cells 2-4).

    Returns what the notebook feeds the layer: an (N, C, k*T, V, 1) float32 tensor.  planar=False: a permuted view of an
    (N, k*T, V, C) buffer -- the notebook's own strides (coordinate axis innermost), so `VirtualRadar.forward` selects the
    same range rounding as the reference does for the notebook.  planar=True: standard-contiguous memory for
    `VirtualRadar.forward_planar_fma`, which skips the layout copy (C ABI vr_pad_frames_joints)."""
    if not isinstance(data, torch.Tensor) or data.dim() not in (3, 4):
        raise ValueError("expected a (T,V,C) or (N,T,V,C) tensor")
    if data.dtype not in (torch.float32, torch.float64):
        raise ValueError("pad_frames_notebook takes float32 or float64; got %s" % data.dtype)
    if not data.is_cuda:
        raise RuntimeError("pad_frames_notebook (B200) has no CPU path: move the array to a CUDA device")
    xb = (data.unsqueeze(0) if data.dim() == 3 else data).contiguous()
    N, T, V, C = xb.shape
    k = int(num_pad_frames)
    out = torch.empty((N, C, k * T, V) if planar else (N, k * T, V, C), dtype=torch.float32, device=data.device)
    if N > 0:
        with torch.cuda.device(data.device):
            stream = torch.cuda.current_stream(data.device).cuda_stream
            rc = _cabi.lib().vr_pad_frames_joints(xb.data_ptr(), 1 if xb.dtype == torch.float64 else 0, N, T, V, C, k,
                                                  ctypes.c_float(float(sigma)), 1 if planar else 0, out.data_ptr(),
                                                  ctypes.c_void_p(stream))
        _cabi.check(rc)
    return out.unsqueeze(-1) if planar else out.permute(0, 3, 1, 2).unsqueeze(-1)
