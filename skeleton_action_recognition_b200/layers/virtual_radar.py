"""Drop-in replacement for the reference's `layers/virtual_radar.py` (class `VirtualRadar`,
module-level `edges`): same constructor arguments, same `forward(x)` signature, same
`state_dict` keys -- but `forward` is one fused sm_100a CUDA kernel reached through the C ABI of
include/virtual_radar_b200.h.  PyTorch is used only for device memory and streams.

Reference behaviour mirrored here (file:line in /root/reference):
  * constructor kwargs and defaults                     layers/virtual_radar.py:36-45
  * parameters `wavelength` (0-d), `radar_location` (3,) layers/virtual_radar.py:65-69
  * `self.src`, `self.dst` python lists                  layers/virtual_radar.py:70
  * `self.stft` with parameters wsin/wcos (n_fft,1,n_fft) layers/virtual_radar.py:71-76 (nnAudio)
  * forward: (N,3,T,V,M) f32 -> (N, n_fft, T//hop+1) f32  layers/virtual_radar.py:79-134

There is no CPU path and no PyTorch fallback: a CPU tensor, a missing shared object or a shape the
kernels do not cover raises.
"""
import ctypes
import functools
import math
import numbers

import numpy as np
import torch

from .. import _cabi

# Default skeleton: the reference's NTU RGB+D bone list (layers/virtual_radar.py:10-13),
# grouped here by limb.  24 bones, 25 joints, 18 distinct source joints.
_SPINE = [(0, 1), (1, 20), (20, 2), (2, 3)]
_LEFT_ARM = [(20, 4), (4, 5), (5, 6), (6, 7), (7, 21), (7, 22)]
_RIGHT_ARM = [(20, 8), (8, 9), (9, 10), (10, 11), (11, 23), (11, 24)]
_HIPS = [(0, 16), (0, 12)]
_LEFT_LEG = [(12, 13), (13, 14), (14, 15)]
_RIGHT_LEG = [(16, 17), (17, 18), (18, 19)]
edges = _SPINE + _LEFT_ARM + _RIGHT_ARM + _HIPS + _LEFT_LEG + _RIGHT_LEG


class _STFTKernels(torch.nn.Module):
    """Holds `wsin` / `wcos` so that `state_dict()` has the reference's `stft.wsin`, `stft.wcos`
    entries (nnAudio 0.1.x STFT parameters; SURVEY Appendix B).  The CUDA path evaluates the
    same windowed DFT with an FFT and does not read these tensors; `assert_dft()` verifies that a
    loaded checkpoint still holds the analytic Hann-windowed Fourier kernels."""

    def __init__(self, n_fft, hop_length, trainable, device):
        super().__init__()
        self.n_fft, self.stride = n_fft, hop_length
        wsin, wcos = self.analytic(n_fft)
        self.wsin = torch.nn.Parameter(wsin.to(device), requires_grad=trainable)
        self.wcos = torch.nn.Parameter(wcos.to(device), requires_grad=trainable)

    @staticmethod
    def analytic(n_fft):
        s = np.arange(n_fft, dtype=np.float64)
        window = 0.5 - 0.5 * np.cos(2 * np.pi * s / n_fft)          # scipy get_window('hann', fftbins=True)
        ang = 2 * np.pi * np.arange(n_fft, dtype=np.float64)[:, None] * s[None, :] / n_fft
        wsin = (window * np.sin(ang)).astype(np.float32)[:, None, :]
        wcos = (window * np.cos(ang)).astype(np.float32)[:, None, :]
        return torch.from_numpy(wsin), torch.from_numpy(wcos)

    def is_dft(self):
        wsin, wcos = self.analytic(self.n_fft)
        return bool(torch.allclose(self.wsin.detach().cpu(), wsin, atol=1e-6)
                    and torch.allclose(self.wcos.detach().cpu(), wcos, atol=1e-6))

    def assert_dft(self):
        if not self.is_dft():
            raise NotImplementedError("stft.wsin/wcos differ from the Hann-windowed Fourier kernels")

    def logmag(self, iq, frames=None):
        """General-kernel path (trained or trainable `wsin`/`wcos`, or an `n_fft` the fused FFT does not cover): what the
        reference computes at layers/virtual_radar.py:124-133 with nnAudio's conv1d STFT, as one float32-accurate GEMM per
        batch on the tensor cores (C ABI vr_stft_general_f32: tcgen05.mma kind::tf32, 3-term split, accumulator in tensor
        memory, magnitude / log / roll in the epilogue), differentiable with respect to `wsin`, `wcos` and `iq`
        (vr_stft_general_backward_f32).  iq (N,T,2) CUDA float32 -> (N, n_fft, T//hop+1).  `frames` (optional): a strictly
        increasing int32 CUDA tensor of frame indices; only those columns are computed (vr_stft_general_frames_f32), bit for
        bit the same, -> (N, n_fft, len(frames))."""
        if not iq.is_cuda:
            raise RuntimeError("the general-kernel STFT (B200) has no CPU path")
        return _GeneralSTFTFunction.apply(iq, self.wsin, self.wcos, self.n_fft, self.stride, torch.is_grad_enabled(), frames)

    def _logmag_torch(self, iq):
        """TEST CROSS-CHECK ONLY (never called by forward): the same computation with torch ops (cuBLAS GEMM + autograd)."""
        n = self.n_fft
        zp = torch.nn.functional.pad(iq.permute(0, 2, 1), (n // 2, n // 2), mode="reflect")       # (N,2,T+n)
        frames = zp.unfold(2, n, self.stride)                                                       # (N,2,F,n)
        wc, ws = self.wcos[:, 0, :].t(), self.wsin[:, 0, :].t()                                     # (n, n_fft)
        c, s_ = torch.matmul(frames, wc), torch.matmul(frames, ws)                                  # (N,2,F,n_fft)
        real = c[:, 0] + s_[:, 1]            # stft(I).real - stft(Q).imag, nnAudio's imag = -conv(x, wsin)
        imag = c[:, 1] - s_[:, 0]            # stft(I).imag + stft(Q).real
        mag = torch.sqrt(real * real + imag * imag)
        out = torch.log(mag + 1e-6).transpose(1, 2)                                                 # (N,n_fft,F)
        return torch.roll(out, n // 2, dims=1)


class _GeneralSTFTFunction(torch.autograd.Function):
    """STFT against general kernels + log-magnitude + roll: forward and backward are the tcgen05 GEMM kernels of
    csrc/vr_stft_gemm.cuh behind vr_stft_general_f32 / vr_stft_general_backward_f32 (no library GEMM, no autograd graph).
    With a frame table, only the listed frames (vr_stft_general_frames_f32 / vr_stft_general_frames_backward_f32)."""

    @staticmethod
    def forward(ctx, iq, wsin, wcos, n_fft, hop, grad_mode, frames=None):
        iq = iq.contiguous()
        if iq.dtype != torch.float32 or wsin.dtype != torch.float32:
            raise ValueError("the general-kernel STFT computes in float32")
        N, T, _ = iq.shape
        L = _cabi.lib()
        parts = (ctypes.c_int64 * 3)()
        if frames is None:
            L.vr_stft_general_workspace_floats(N, T, n_fft, hop, parts)
            ncols = T // hop + 1
        else:
            ncols = frames.numel()
            L.vr_stft_general_frames_workspace_floats(N, ncols, n_fft, parts)
        dev = iq.device
        work = torch.empty(max(int(parts[0]), 1), dtype=torch.float32, device=dev)       # the padded signal / the kept frames
        bt = torch.empty(max(int(parts[1]), 1), dtype=torch.float32, device=dev)
        # needs_input_grad ignores torch.no_grad(): the caller passes the grad mode, so that inference does not write Re / Im
        need = bool(grad_mode) and any(ctx.needs_input_grad[:3])
        csave = torch.empty(max(int(parts[2]), 1), dtype=torch.float32, device=dev) if need else None
        out = torch.empty((N, n_fft, ncols), dtype=torch.float32, device=dev)
        if N > 0:
            with torch.cuda.device(dev):
                stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
                args = (wsin.contiguous().data_ptr(), wcos.contiguous().data_ptr(), work.data_ptr(), bt.data_ptr(),
                        csave.data_ptr() if need else None, out.data_ptr(), stream)
                if frames is None:
                    rc = L.vr_stft_general_f32(iq.data_ptr(), N, T, n_fft, hop, *args)
                else:
                    rc = L.vr_stft_general_frames_f32(iq.data_ptr(), N, T, n_fft, hop, frames.data_ptr(), ncols, *args)
            _cabi.check(rc)
        if need:
            ctx.save_for_backward(work, bt, csave, frames)
        ctx.dims = (N, T, n_fft, hop, ncols, tuple(wsin.shape))
        return out

    @staticmethod
    def backward(ctx, gout):
        work, bt, csave, frames = ctx.saved_tensors
        N, T, n_fft, hop, ncols, wshape = ctx.dims
        dev = gout.device
        need_iq, need_w = ctx.needs_input_grad[0], (ctx.needs_input_grad[1] or ctx.needs_input_grad[2])
        g = gout.contiguous().to(torch.float32)
        dc = torch.empty_like(csave)
        da = torch.empty(N * ncols * 2 * n_fft, dtype=torch.float32, device=dev) if need_iq else None   # frame gradients
        dbt = torch.empty_like(bt) if need_w else None
        giq = torch.empty((N, T, 2), dtype=torch.float32, device=dev) if need_iq else None
        gsin = torch.empty(wshape, dtype=torch.float32, device=dev) if need_w else None
        gcos = torch.empty(wshape, dtype=torch.float32, device=dev) if need_w else None
        if N > 0:
            ptr = lambda t: t.data_ptr() if t is not None else None     # noqa: E731
            with torch.cuda.device(dev):
                stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
                outs = (dc.data_ptr(), ptr(da), ptr(dbt), ptr(giq), ptr(gsin), ptr(gcos), stream)
                if frames is None:
                    rc = _cabi.lib().vr_stft_general_backward_f32(g.data_ptr(), work.data_ptr(), bt.data_ptr(), csave.data_ptr(),
                                                                  N, T, n_fft, hop, *outs)
                else:
                    rc = _cabi.lib().vr_stft_general_frames_backward_f32(g.data_ptr(), work.data_ptr(), bt.data_ptr(),
                                                                         csave.data_ptr(), N, T, n_fft, hop,
                                                                         frames.data_ptr(), ncols, *outs)
            _cabi.check(rc)
        return (giq, gsin if ctx.needs_input_grad[1] else None, gcos if ctx.needs_input_grad[2] else None, None, None, None, None)


def _param_grad_buffer(flags, N, T, device):
    """float64 gradient buffer of a backward call: the 4 batch-summed gradients, or with VR_FLAG_PER_SEQUENCE N x 4
    per-sequence gradients followed by the scratch of their reduction (T: the steps the adjoint runs over)."""
    if flags & _cabi.VR_FLAG_PER_SEQUENCE:
        return torch.zeros(_cabi.per_sequence_grad_doubles(N, T), dtype=torch.float64, device=device)
    return torch.zeros(4, dtype=torch.float64, device=device)


def _param_grads(ctx, gp, lam, loc):
    """(dL/dwavelength, dL/dradar_location) in the shapes of `lam` and `loc` -- () and (3,), or (N,) and (N, 3) -- from the
    buffer of _param_grad_buffer; None where no gradient is needed."""
    g = gp[:4 * lam.numel()].view(-1, 4)
    g_lam = g[:, 0].to(torch.float32).reshape(lam.shape) if ctx.needs_input_grad[0] else None
    g_loc = g[:, 1:4].to(torch.float32).reshape(loc.shape) if ctx.needs_input_grad[1] else None
    return g_lam, g_loc


class _RadarFunction(torch.autograd.Function):
    """forward() with gradients for `wavelength`, `radar_location` and `x` (the reference gets them from
    PyTorch autograd over layers/virtual_radar.py:79-134; here: C ABI vr_backward_f32).  The
    forward launch is the same fused kernel, asked to also save the complex baseband signal."""

    @staticmethod
    def forward(ctx, lam, loc, xc, layer, flags, noise=None):
        out, iq = layer._launch(xc, flags, want_iq=True, lam=lam, loc=loc, noise=noise)
        ctx.save_for_backward(lam, loc, xc, iq)      # iq carries the receiver noise: the STFT adjoint reads log|z + xi|
        ctx.layer, ctx.flags = layer, flags & ~_cabi.VR_FLAG_NOISE
        return out

    @staticmethod
    def backward(ctx, grad_out):
        lam, loc, xc, iq = ctx.saved_tensors
        layer = ctx.layer
        _, _, T, V, M = xc.shape
        N = xc.shape[0] * _cabi.views_of(ctx.flags)        # outputs: R views of each x sequence (VR_FLAG_VIEWS)
        g = grad_out.contiguous().to(torch.float32)
        gz = torch.empty((N, T, 2), dtype=torch.float32, device=xc.device)
        gp = _param_grad_buffer(ctx.flags, N, T, xc.device)
        gx = torch.empty_like(xc) if ctx.needs_input_grad[2] else None
        with torch.cuda.device(xc.device):
            stream = torch.cuda.current_stream(xc.device).cuda_stream
            rc = _cabi.lib().vr_backward_f32(xc.data_ptr(), iq.data_ptr(), g.data_ptr(), N, T, V, M,
                                             layer._src_c, layer._dst_c, len(layer.src),
                                             lam.data_ptr(), loc.data_ptr(), layer.n_fft, layer.hop_length,
                                             ctx.flags, gz.data_ptr(), gp.data_ptr(),
                                             gx.data_ptr() if gx is not None else None, ctypes.c_void_p(stream))
        _cabi.check(rc)
        g_lam, g_loc = _param_grads(ctx, gp, lam, loc)
        return g_lam, g_loc, gx, None, None, None


class _SynthFunction(torch.autograd.Function):
    """Complex baseband synthesis only (layers/virtual_radar.py:93-123) -> iq (N,T,2), with gradients for
    `wavelength`, `radar_location` and `x` (C ABI vr_synth_adjoint_f32).  Used when the STFT is a general,
    trainable kernel pair and therefore runs outside the fused kernel."""

    @staticmethod
    def forward(ctx, lam, loc, xc, layer, flags, noise=None):
        iq = layer._synth(xc, flags, lam, loc, noise)
        ctx.save_for_backward(lam, loc, xc)
        ctx.layer, ctx.flags = layer, flags & ~_cabi.VR_FLAG_NOISE     # d(z + xi)/d(theta) = dz/d(theta)
        return iq

    @staticmethod
    def backward(ctx, grad_iq):
        lam, loc, xc = ctx.saved_tensors
        layer = ctx.layer
        _, _, T, V, M = xc.shape
        N = xc.shape[0] * _cabi.views_of(ctx.flags)
        g = grad_iq.contiguous().to(torch.float32)
        gp = _param_grad_buffer(ctx.flags, N, T, xc.device)
        gx = torch.empty_like(xc) if ctx.needs_input_grad[2] else None
        with torch.cuda.device(xc.device):
            stream = torch.cuda.current_stream(xc.device).cuda_stream
            rc = _cabi.lib().vr_synth_adjoint_f32(xc.data_ptr(), g.data_ptr(), N, T, V, M, layer._src_c, layer._dst_c,
                                                  len(layer.src), lam.data_ptr(), loc.data_ptr(), ctx.flags, gp.data_ptr(),
                                                  gx.data_ptr() if gx is not None else None, ctypes.c_void_p(stream))
        _cabi.check(rc)
        g_lam, g_loc = _param_grads(ctx, gp, lam, loc)
        return g_lam, g_loc, gx, None, None, None


class _UpsampledRadarFunction(torch.autograd.Function):
    """forward_upsampled() with gradients for `wavelength` and `radar_location`, without the up-sampled batch: the forward
    is the fused up-sampling + radar launch, asked to also save the complex baseband signal (vr_forward_upsampled_debug_f32);
    the spline's per-interval cubics stay in the workspace, from which the backward (vr_backward_upsampled_params_f32)
    re-evaluates the joint positions of every up-sampled step."""

    @staticmethod
    def forward(ctx, lam, loc, xc, layer, k, sigma, flags=0, noise=None):
        _, _, T, V, M = xc.shape
        N = xc.shape[0] * _cabi.views_of(flags)             # outputs; the spline is solved once per raw sequence
        L = _cabi.lib()
        nbytes = int(L.vr_upsampled_workspace_bytes(xc.shape[0], T, V, M))
        work = torch.empty(max(nbytes, 8) // 8, dtype=torch.float64, device=xc.device)
        out = torch.empty((N, layer.n_fft, (k * T) // layer.hop_length + 1), dtype=torch.float32, device=xc.device)
        iq = torch.empty((N, k * T, 2), dtype=torch.float32, device=xc.device)
        with torch.cuda.device(xc.device):
            stream = ctypes.c_void_p(torch.cuda.current_stream(xc.device).cuda_stream)
            _set_noise(noise)
            rc = L.vr_forward_upsampled_debug_f32(xc.data_ptr(), N, T, V, M, layer._src_c, layer._dst_c, len(layer.src),
                                                  lam.data_ptr(), loc.data_ptr(), layer.n_fft, layer.hop_length, flags,
                                                  k, ctypes.c_float(float(sigma)), work.data_ptr(), nbytes,
                                                  out.data_ptr(), iq.data_ptr(), stream)
        _cabi.check(rc)
        ctx.save_for_backward(lam, loc, work, iq)      # iq carries the receiver noise, as in _RadarFunction
        ctx.layer, ctx.dims, ctx.flags = layer, (N, T, V, M, k), flags & ~_cabi.VR_FLAG_NOISE
        return out

    @staticmethod
    def backward(ctx, grad_out):
        lam, loc, work, iq = ctx.saved_tensors
        layer = ctx.layer
        N, T, V, M, k = ctx.dims
        g = grad_out.contiguous().to(torch.float32)
        gz = torch.empty_like(iq)
        gp = _param_grad_buffer(ctx.flags, N, k * T, iq.device)
        with torch.cuda.device(iq.device):
            stream = torch.cuda.current_stream(iq.device).cuda_stream
            rc = _cabi.lib().vr_backward_upsampled_params_f32(work.data_ptr(), iq.data_ptr(), g.data_ptr(), N, T, V, M,
                                                              layer._src_c, layer._dst_c, len(layer.src),
                                                              lam.data_ptr(), loc.data_ptr(), layer.n_fft, layer.hop_length,
                                                              ctx.flags, k, gz.data_ptr(), gp.data_ptr(), ctypes.c_void_p(stream))
        _cabi.check(rc)
        g_lam, g_loc = _param_grads(ctx, gp, lam, loc)
        return g_lam, g_loc, None, None, None, None, None, None


class _UpsampledSynthFunction(torch.autograd.Function):
    """Complex baseband synthesis of the up-sampled batch -> iq (N, k*T, 2), with gradients for `wavelength` and
    `radar_location`, without the up-sampled batch: the forward (vr_synth_upsampled_f32) leaves the spline's per-interval
    cubics in the workspace, from which the backward (vr_synth_adjoint_upsampled_f32) re-evaluates the joint positions.
    Used by forward_upsampled when the STFT is general and therefore runs outside the fused kernel."""

    @staticmethod
    def forward(ctx, lam, loc, xc, layer, k, sigma, flags=0, noise=None):
        iq, work = layer._synth_upsampled(xc, k, sigma, lam, loc, flags, noise)
        ctx.save_for_backward(lam, loc, work)
        ctx.layer, ctx.dims, ctx.flags = layer, (iq.shape[0],) + tuple(xc.shape[1:]) + (k,), flags & ~_cabi.VR_FLAG_NOISE
        return iq

    @staticmethod
    def backward(ctx, grad_iq):
        lam, loc, work = ctx.saved_tensors
        layer = ctx.layer
        N, _, T, V, M, k = ctx.dims
        g = grad_iq.contiguous().to(torch.float32)
        gp = _param_grad_buffer(ctx.flags, N, k * T, g.device)
        with torch.cuda.device(g.device):
            stream = torch.cuda.current_stream(g.device).cuda_stream
            rc = _cabi.lib().vr_synth_adjoint_upsampled_f32(work.data_ptr(), g.data_ptr(), N, T, V, M, layer._src_c, layer._dst_c,
                                                            len(layer.src), lam.data_ptr(), loc.data_ptr(), ctx.flags, k,
                                                            gp.data_ptr(), ctypes.c_void_p(stream))
        _cabi.check(rc)
        g_lam, g_loc = _param_grads(ctx, gp, lam, loc)
        return g_lam, g_loc, None, None, None, None, None, None


def _set_noise(noise):
    """vr_set_noise right before a launch that carries VR_FLAG_NOISE; noise: (std, seed) of _noise, or None."""
    if noise is not None:
        _cabi.set_noise(*noise)


def kept_frame_table(n_frames, image_size):
    """The frames a nearest resize of `n_frames` spectrogram columns to `image_size` reads, by ATen's rule (column c reads
    min(int(floorf(c * scale)), n_frames - 1), scale = float32(n_frames) / image_size): an int32 array of `image_size`
    strictly increasing indices when n_frames > image_size, else None (every frame is read; the full STFT is computed)."""
    if n_frames <= image_size:
        return None
    scale = np.float32(n_frames) / np.float32(image_size)
    idx = np.minimum(np.floor(np.arange(image_size, dtype=np.float32) * scale).astype(np.int64), n_frames - 1)
    if not (np.diff(idx) > 0).all():
        raise AssertionError("nearest map from %d columns to %d frames is not strictly increasing" % (image_size, n_frames))
    return idx.astype(np.int32)


@functools.lru_cache(maxsize=64)
def _kept_frames_on(n_frames, image_size, device):
    return torch.from_numpy(kept_frame_table(n_frames, image_size)).to(device)


class VirtualRadar(torch.nn.Module):
    """Skeleton sequences -> micro-Doppler log-spectrograms on a B200 (see module docstring)."""

    def __init__(self, edges=edges, wavelength=1e-3, radar_location=[0., 0., 0.],
                 train_wavelength=False, train_radar_location=False, train_stft_kernel=False,
                 n_fft=256, hop_length=16, device='cuda:0'):
        super().__init__()
        _cabi.lib()   # fail at construction time if the extension is missing
        self.wavelength = torch.nn.Parameter(torch.as_tensor(wavelength, dtype=torch.float32),
                                             requires_grad=bool(train_wavelength))
        self.radar_location = torch.nn.Parameter(torch.as_tensor(radar_location, dtype=torch.float32),
                                                 requires_grad=bool(train_radar_location))
        self.src, self.dst = map(list, zip(*edges))
        self.stft = _STFTKernels(n_fft, hop_length, bool(train_stft_kernel), device)
        self.n_fft = n_fft
        self.hop_length = hop_length
        self._src_c = _cabi.i32_array(self.src)
        self._dst_c = _cabi.i32_array(self.dst)
        # Opt-in for streams of INDEPENDENT batches (VR_FLAG_INPUTS_READY): set True only if the kernel launched just
        # before each forward on the same stream neither produces x nor touches the output; consecutive forwards then
        # overlap (a batch starts in the SM slots the previous one has vacated).  Default: plain stream order.
        self.assume_inputs_ready = False
        # Profiling aid: True wraps every launch of this layer in an NVTX range ("VirtualRadar.<entry>") so that timeline
        # tools show the fused stage among the model's other kernels (SURVEY 5: tracing hooks).  Off by default.
        self.nvtx_ranges = False

    # the ctypes arrays are not picklable / deep-copyable (DataParallel.replicate copies __dict__)
    def __getstate__(self):
        d = self.__dict__.copy()
        d.pop("_src_c", None)
        d.pop("_dst_c", None)
        d.pop("_host_params", None)
        return d

    def __setstate__(self, d):
        self.__dict__.update(d)
        self._src_c = _cabi.i32_array(self.src)
        self._dst_c = _cabi.i32_array(self.dst)

    def _check_stft(self):
        """The fused kernel evaluates the analytic Hann-windowed DFT with an FFT.  Trained `stft.wsin/wcos` (reference
        `train_stft_kernel=True`, or a checkpoint of such a model) must never silently be replaced by it, so the
        parameters are compared with the analytic kernels (one small device-to-host copy) whenever they may have
        changed: the verdict is cached against the tensors' identity and version counters, which every in-place
        update through the parameters -- optimizer step, `load_state_dict`, `wsin.copy_()`, `.to()` -- changes.  (Writes
        through `wsin.data` bypass PyTorch's version counters; call `invalidate_stft_cache()` after such an edit.)"""
        if getattr(self, "_stft_trusted", False):       # a DataParallel replica: the parent module has just checked
            return
        key = tuple((t.data_ptr(), t._version, t.device) for t in (self.stft.wsin, self.stft.wcos))
        if getattr(self, "_stft_key", None) != key:
            self._stft_is_dft = self.stft.is_dft()
            self._stft_key = key

    def invalidate_stft_cache(self):
        self._stft_key = None

    def _replicate_for_data_parallel(self):
        if not (self.stft.wsin.requires_grad or self.stft.wcos.requires_grad):
            self._check_stft()                          # once on the parent instead of once per replica and forward
        replica = super()._replicate_for_data_parallel()
        replica._stft_trusted = True
        return replica

    def _general_stft(self):
        """True -> CUDA synthesis, then the STFT against `wsin`/`wcos` as they are (`_STFTKernels.logmag`).  Trainable
        kernels always take this path, with or without grad mode: an eval pass of a model being trained must see the
        kernels the optimizer has produced."""
        if self.stft.wsin.requires_grad or self.stft.wcos.requires_grad or self.n_fft != self._FUSED_N_FFT:
            return True
        self._check_stft()
        return not self._stft_is_dft

    def output_shape(self, x_shape):
        return (x_shape[0], self.n_fft, x_shape[2] // self.hop_length + 1)

    def _check_input(self, x):
        if not isinstance(x, torch.Tensor) or x.dim() != 5 or x.shape[1] != 3:
            raise ValueError("expected x of shape (batch, 3, timesteps, vertices, num_graphs), got %s"
                             % (tuple(x.shape) if isinstance(x, torch.Tensor) else type(x),))
        if x.dtype != torch.float32:
            raise ValueError("VirtualRadar computes in float32 like the reference; got %s" % x.dtype)

    def _check_device(self, x):
        if not x.is_cuda:
            raise RuntimeError("VirtualRadar (B200) has no CPU path: move x to a CUDA device, or call "
                               "forward_host(x) to stream a pinned host batch through the GPU")
        lam, loc = self.wavelength, self.radar_location
        if lam.device != x.device or loc.device != x.device:
            raise RuntimeError("module parameters are on %s but x is on %s; call .to(x.device)" % (lam.device, x.device))
        return lam, loc

    def _placements(self, x, radar_location, wavelength, noise_std=None, noise_seed=None):
        """Per-sequence radar placements (the `radar_location=` / `wavelength=` keywords of forward, forward_image and
        forward_upsampled) and receiver noise (`noise_std=` / `noise_seed=`) -> None when none is given, else
        (wavelength (N,), radar_location (N, 3), flags, noise): each placement keyword expanded to the batch and made
        contiguous, the module parameter standing in for a keyword not given.  Autograd's expand carries the
        per-sequence gradients back to whatever the caller passed (summed where it broadcast).  flags: what the launch
        adds (VR_FLAG_PER_SEQUENCE, and VR_FLAG_NOISE with noise); noise: (std (N,), seed) of _noise, or None."""
        noise = self._noise(x, noise_std, noise_seed, (x.shape[0],))
        if radar_location is None and wavelength is None and noise is None:
            return None
        N = x.shape[0]
        lam = self._expand_placement(x, "wavelength", wavelength, self.wavelength, (N,))
        loc = self._expand_placement(x, "radar_location", radar_location, self.radar_location, (N, 3))
        return lam, loc, _cabi.VR_FLAG_PER_SEQUENCE | (_cabi.VR_FLAG_NOISE if noise is not None else 0), noise

    def _view_placements(self, x, radar_location, wavelength, noise_std=None, noise_seed=None):
        """The placements of forward_views -> (wavelength (N R,), radar_location (N R, 3), flags, noise): R from
        radar_location's second-to-last dimension, each keyword expanded to (N, R[, 3]) and flattened view-minor (output
        n R + r is view r of sequence n), the module's wavelength standing in for `wavelength=None`; noise_std likewise
        from (N, R).  flags: VR_FLAG_PER_SEQUENCE | VR_FLAG_VIEWS(R) [| VR_FLAG_NOISE]."""
        if not isinstance(radar_location, torch.Tensor) or radar_location.dim() < 2:
            raise ValueError("radar_location must be a tensor of R placements, (R, 3) for every sequence or (N, R, 3), got %s"
                             % (tuple(radar_location.shape) if isinstance(radar_location, torch.Tensor) else type(radar_location),))
        N, R = x.shape[0], radar_location.shape[-2]
        if not 1 <= R <= 255:
            raise ValueError("forward_views takes 1 to 255 views per sequence, got R=%d (radar_location of shape %s)"
                             % (R, tuple(radar_location.shape)))
        lam = self._expand_placement(x, "wavelength", wavelength, self.wavelength, (N, R))
        loc = self._expand_placement(x, "radar_location", radar_location, self.radar_location, (N, R, 3))
        noise = self._noise(x, noise_std, noise_seed, (N, R))
        flags = _cabi.VR_FLAG_PER_SEQUENCE | _cabi.views_flag(R) | (_cabi.VR_FLAG_NOISE if noise is not None else 0)
        return lam.reshape(N * R), loc.reshape(N * R, 3), flags, noise

    @staticmethod
    def _noise(x, noise_std, noise_seed, shape):
        """The receiver-noise keywords -> None without `noise_std`, else (std, seed): std the float32 noise standard
        deviations broadcast to `shape` and flattened (one per output), seed a 0-d int64 tensor on x's device holding the
        64 seed bits -- `noise_seed` itself when it is such a tensor (what a CUDA graph should pass: the launch reads it
        at replay time), a Python int in [0, 2**64) copied to the device, or None: drawn from torch's CUDA generator, so
        every call has fresh noise and torch.manual_seed makes the sequence of calls reproducible.  A float level must be
        finite and non-negative; a tensor's values are not checked (that would synchronise with the device): a negative
        level gives noise of its magnitude, a NaN level NaN outputs."""
        if noise_std is None:
            if noise_seed is not None:
                raise ValueError("noise_seed needs noise_std: the noise level of every output")
            return None
        if isinstance(noise_std, torch.Tensor):
            if noise_std.requires_grad:
                raise ValueError("noise_std must not require grad: the layer has no gradient with respect to the noise level")
            std = VirtualRadar._expand_placement(x, "noise_std", noise_std, None, shape)
        elif isinstance(noise_std, numbers.Real) and not isinstance(noise_std, bool):
            v = float(noise_std)
            if not (math.isfinite(v) and v >= 0):
                raise ValueError("noise_std must be a finite non-negative noise standard deviation, got %r" % (noise_std,))
            std = torch.full(shape, v, dtype=torch.float32, device=x.device)
        else:
            raise ValueError("noise_std must be a float or a float32 tensor that broadcasts to %s, got %s"
                             % (shape, type(noise_std)))
        if noise_seed is None:
            seed = torch.randint(0, 2 ** 63 - 1, (), dtype=torch.int64, device=x.device)
        elif isinstance(noise_seed, torch.Tensor):
            if noise_seed.dtype != torch.int64 or noise_seed.dim() != 0:
                raise ValueError("noise_seed must be an int or a 0-d int64 tensor, got a %s tensor of shape %s"
                                 % (noise_seed.dtype, tuple(noise_seed.shape)))
            if noise_seed.device != x.device:
                raise RuntimeError("noise_seed is on %s but x is on %s: the seed is read on x's device"
                                   % (noise_seed.device, x.device))
            seed = noise_seed
        elif isinstance(noise_seed, numbers.Integral) and not isinstance(noise_seed, bool):
            s = int(noise_seed)
            if not 0 <= s < 2 ** 64:
                raise ValueError("noise_seed must be in [0, 2**64), got %d" % s)
            # a fill kernel, not a pageable host-to-device copy: no stream synchronisation per call
            seed = torch.full((), s - 2 ** 64 if s >= 2 ** 63 else s, dtype=torch.int64, device=x.device)
        else:
            raise ValueError("noise_seed must be an int or a 0-d int64 tensor, got %s" % type(noise_seed))
        return std.reshape(-1), seed

    @staticmethod
    def _expand_placement(x, name, value, param, shape):
        """One placement keyword checked (float32, on x's device) and expanded to `shape`, contiguous; `param` if None."""
        if value is None:
            value = param
        elif not isinstance(value, torch.Tensor) or value.dtype != torch.float32:
            raise ValueError("%s must be a float32 tensor that broadcasts to %s, got %s"
                             % (name, shape, value.dtype if isinstance(value, torch.Tensor) else type(value)))
        elif not value.is_cuda or value.device != x.device:
            raise RuntimeError("%s is on %s but x is on %s: per-sequence placements are read on x's device"
                               % (name, value.device, x.device))
        if tuple(value.shape) != shape or not value.is_contiguous():   # (a full contiguous tensor is used as it is)
            try:
                value = value.expand(shape)
            except RuntimeError:
                raise ValueError("%s of shape %s does not broadcast to %s" % (name, tuple(value.shape), shape)) from None
            value = value.contiguous()
        return value

    def _prepare(self, x):
        """Pick the range rounding mode from the caller's strides BEFORE normalising the layout
        (SURVEY fact 6: ATen's CPU norm rounds differently when the coordinate axis is innermost)."""
        flags = _cabi.VR_FLAG_RANGE_FMA if x.stride(1) == 1 and x.shape[1] > 1 else 0
        return x.contiguous(), flags

    _FUSED_N_FFT = 256      # the fused kernel's FFT size; other n_fft values go through the general-kernel path

    def _launch(self, xc, flags, want_iq=False, lam=None, loc=None, noise=None):
        """One fused launch.  lam / loc: the radar parameters to read (default: the module's; (N,) and (N, 3) with
        VR_FLAG_PER_SEQUENCE in flags, N = R x the rows of xc with VR_FLAG_VIEWS(R)); noise: with VR_FLAG_NOISE."""
        _, _, T, V, M = xc.shape
        N = xc.shape[0] * _cabi.views_of(flags)
        lam = self.wavelength if lam is None else lam
        loc = self.radar_location if loc is None else loc
        n_fft = self._FUSED_N_FFT if want_iq else self.n_fft       # iq does not depend on the STFT parameters
        if self.assume_inputs_ready:
            flags |= _cabi.VR_FLAG_INPUTS_READY
        out = torch.empty((N, n_fft, T // self.hop_length + 1), dtype=torch.float32, device=xc.device)
        iq = torch.empty((N, T, 2), dtype=torch.float32, device=xc.device) if want_iq else None
        if N == 0:
            return out, iq
        L = _cabi.lib()
        if self.nvtx_ranges:
            torch.cuda.nvtx.range_push("VirtualRadar.forward%s N=%d T=%d" % ("+iq" if want_iq else "", N, T))
        try:
            with torch.cuda.device(xc.device):
                stream = ctypes.c_void_p(torch.cuda.current_stream(xc.device).cuda_stream)
                args = (xc.data_ptr(), N, T, V, M, self._src_c, self._dst_c, len(self.src), lam.data_ptr(),
                        loc.data_ptr(), n_fft, self.hop_length, flags, out.data_ptr())
                _set_noise(noise)
                rc = L.vr_forward_debug_f32(*args, iq.data_ptr(), stream) if want_iq else L.vr_forward_f32(*args, stream)
        finally:
            if self.nvtx_ranges:
                torch.cuda.nvtx.range_pop()
        _cabi.check(rc)
        return out, iq

    def _synth(self, xc, flags, lam=None, loc=None, noise=None):
        """Synthesis only (C ABI vr_synth_f32): the complex baseband signal (N,T,2) that the general-kernel STFT reads,
        bit for bit forward_debug's, without any STFT work."""
        _, _, T, V, M = xc.shape
        N = xc.shape[0] * _cabi.views_of(flags)
        lam = self.wavelength if lam is None else lam
        loc = self.radar_location if loc is None else loc
        if self.assume_inputs_ready:
            flags |= _cabi.VR_FLAG_INPUTS_READY
        iq = torch.empty((N, T, 2), dtype=torch.float32, device=xc.device)
        if N == 0:
            return iq
        if self.nvtx_ranges:
            torch.cuda.nvtx.range_push("VirtualRadar.synth N=%d T=%d" % (N, T))
        try:
            with torch.cuda.device(xc.device):
                stream = ctypes.c_void_p(torch.cuda.current_stream(xc.device).cuda_stream)
                _set_noise(noise)
                rc = _cabi.lib().vr_synth_f32(xc.data_ptr(), N, T, V, M, self._src_c, self._dst_c, len(self.src),
                                              lam.data_ptr(), loc.data_ptr(), flags, iq.data_ptr(), stream)
        finally:
            if self.nvtx_ranges:
                torch.cuda.nvtx.range_pop()
        _cabi.check(rc)
        return iq

    def _synth_upsampled(self, xc, k, sigma, lam=None, loc=None, flags=0, noise=None):
        """Synthesis of pad_frames(xc, k, sigma) without the up-sampled batch (C ABI vr_synth_upsampled_f32) -> iq
        (N, k*T, 2) and the workspace holding the spline's cubics.  The up-sampled tensor the reference's loader builds
        is standard-contiguous: range rounding mode "seq" (no VR_FLAG_RANGE_FMA)."""
        _, _, T, V, M = xc.shape
        N = xc.shape[0] * _cabi.views_of(flags)
        lam = self.wavelength if lam is None else lam
        loc = self.radar_location if loc is None else loc
        L = _cabi.lib()
        nbytes = int(L.vr_upsampled_workspace_bytes(xc.shape[0], T, V, M))
        work = torch.empty(max(nbytes, 8) // 8, dtype=torch.float64, device=xc.device)
        iq = torch.empty((N, k * T, 2), dtype=torch.float32, device=xc.device)
        if N == 0:
            return iq, work
        with torch.cuda.device(xc.device):
            stream = ctypes.c_void_p(torch.cuda.current_stream(xc.device).cuda_stream)
            _set_noise(noise)
            rc = L.vr_synth_upsampled_f32(xc.data_ptr(), N, T, V, M, self._src_c, self._dst_c, len(self.src),
                                          lam.data_ptr(), loc.data_ptr(), flags, k,
                                          ctypes.c_float(float(sigma)), work.data_ptr(), nbytes, iq.data_ptr(), stream)
        _cabi.check(rc)
        return iq, work

    def _check_general_length(self, T):
        if T <= max(self.n_fft, self._FUSED_N_FFT) // 2:
            raise ValueError("T=%d must exceed n_fft/2=%d: reflect padding needs it" % (T, max(self.n_fft, self._FUSED_N_FFT) // 2))

    def _general_image(self, iq, image_size):
        """`F.interpolate(self.stft.logmag(iq).unsqueeze(1), image_size)` (nearest) bit for bit.  When the spectrogram has
        more frames than the image has columns, the resize reads exactly `image_size` distinct frames: only those are
        transformed (kept-frames STFT), and resizing the compact spectrogram -- column scale 1 -- reads each once."""
        n_frames = iq.shape[1] // self.hop_length + 1
        frames = _kept_frames_on(n_frames, image_size, iq.device) if n_frames > image_size else None
        return torch.nn.functional.interpolate(self.stft.logmag(iq, frames).unsqueeze(1), image_size)

    def _needs_grad(self, x=None, pl=None):
        if pl is not None:      # per-sequence placements: whatever the caller passed (or the module parameters) decides
            return torch.is_grad_enabled() and (pl[0].requires_grad or pl[1].requires_grad
                                                or (x is not None and x.requires_grad))
        return torch.is_grad_enabled() and (self.wavelength.requires_grad or self.radar_location.requires_grad
                                            or (x is not None and x.requires_grad))

    def forward(self, x, radar_location=None, wavelength=None, noise_std=None, noise_seed=None):
        """x (N,3,T,V,M) -> (N, n_fft, T//hop+1).  `radar_location` / `wavelength` (optional): one radar placement per
        sequence, float32 tensors on x's device that broadcast to (N, 3) and (N,) -- sequence n is seen from
        radar_location[n] at wavelength[n] (C ABI VR_FLAG_PER_SEQUENCE); a keyword not given is the module parameter.
        Differentiable per sequence: the gradients reach the tensors passed (through autograd's expand).  Under
        torch.nn.DataParallel pass full (N, 3) / (N,) tensors: DataParallel splits every tensor argument along dim 0 like
        the batch, so a broadcast-shaped one -- a (3,) location, a 0-d wavelength -- would reach the replicas cut apart
        (expand it to the batch first, e.g. `loc.expand(len(x), 3)`).

        `noise_std` / `noise_seed` (optional): receiver noise (C ABI VR_FLAG_NOISE, DESIGN §3i), a complex Gaussian
        sample xi[n, t] with E|xi|^2 = noise_std[n]^2 added to the baseband of sequence n at every step t before the STFT.
        `noise_std`: a float or a float32 tensor on x's device that broadcasts to (N,), in the units of the I/Q (an
        absolute level, not an SNR); it has no gradient, and a tensor's values are not checked.  `noise_seed`: an int in [0, 2**64), a 0-d int64 CUDA tensor
        (for CUDA graphs: the seed is read when the graph replays), or None (drawn from torch's CUDA generator).  xi
        depends only on (seed, n, t), n the position in this call's batch: a DataParallel replica or a sharded_forward
        rank numbers its own shard from 0, so its noise differs from a single-device call with the same seed.  The
        gradients with respect to x and the placements are those of the noisy spectrogram."""
        self._check_input(x)
        self._check_device(x)
        pl = self._placements(x, radar_location, wavelength, noise_std, noise_seed)
        xc, flags = self._prepare(x)
        return self._run(x, xc, flags, pl)

    def _run(self, x, xc, flags, pl=None):
        """forward() after the layout has been normalised: xc standard-contiguous, flags carry the range rounding mode;
        pl: per-sequence placements (_placements, _view_placements) or None."""
        lam, loc, noise = self.wavelength, self.radar_location, None
        if pl is not None:
            lam, loc, pflags, noise = pl
            flags |= pflags
        if self._general_stft():     # trained / trainable STFT kernels: synthesis on our kernels, STFT as a GEMM
            self._check_general_length(xc.shape[2])
            if xc.shape[0] == 0:
                return self._launch(xc, flags, lam=lam, loc=loc, noise=noise)[0]
            return self.stft.logmag(self._general_iq(x, xc, flags, pl))
        if self._needs_grad(x, pl) and xc.shape[0] > 0:
            return _RadarFunction.apply(lam, loc, xc, self, flags, noise)
        return self._launch(xc, flags, lam=lam, loc=loc, noise=noise)[0]

    def _general_iq(self, x, xc, flags, pl=None):
        lam, loc, noise = self.wavelength, self.radar_location, None
        if pl is not None:
            lam, loc, pflags, noise = pl
            flags |= pflags
        if self._needs_grad(x, pl):
            return _SynthFunction.apply(lam, loc, xc, self, flags, noise)
        return self._synth(xc, flags, lam, loc, noise)

    def forward_notebook(self, data, num_pad_frames=1, sigma=3):
        """virtual_radar_example.ipynb cells 2-4 on the device: `data` is one body's (T, V, 3) array (or a batch
        (N, T, V, 3)), float64 or float32 CUDA tensor.  Equals
        `self(torch.Tensor(np.expand_dims(utils.pad_frames(data, num_pad_frames, sigma).transpose(2, 0, 1), [0, -1])))`
        of the reference (utils.py:82-89 + layers/virtual_radar.py:79-134): the up-sampling kernel writes float32 straight
        in the layer's layout (C ABI vr_pad_frames_joints, planar), and the launch is told to round the radar range the way
        the reference does for the notebook's coordinate-innermost tensor (VR_FLAG_RANGE_FMA) -- no layout copy of the
        k-times larger array in between."""
        from ..upsample import pad_frames_notebook
        if isinstance(data, torch.Tensor) and data.shape[-1] != 3:
            raise ValueError("expected (T, V, 3) or (N, T, V, 3) joint positions, got %s" % (tuple(data.shape),))
        x = pad_frames_notebook(data, num_pad_frames, sigma, planar=True)
        self._check_input(x)
        self._check_device(x)
        return self._run(x, x, _cabi.VR_FLAG_RANGE_FMA)

    def forward_image(self, x, image_size=256, radar_location=None, wavelength=None, noise_std=None, noise_seed=None):
        """The layer fused with its consumer's input stage (reference models/resnet.py:24-26):
        equals `F.interpolate(self(x).unsqueeze(1), image_size)` (nearest) bit for bit, in one launch
        that writes (N, 1, image_size, image_size) directly and transforms only the frames the
        resize keeps.  `radar_location` / `wavelength`: per-sequence placements, and `noise_std` / `noise_seed`
        receiver noise, as in forward()."""
        self._check_input(x)
        self._check_device(x)
        return self._image(x, image_size, self._placements(x, radar_location, wavelength, noise_std, noise_seed))

    def _image(self, x, image_size, pl):
        """forward_image after the input checks; pl: placements (_placements, _view_placements) or None."""
        lam, loc = self.wavelength, self.radar_location
        image_size = int(image_size)
        if image_size < 1:
            raise ValueError("image_size must be positive, got %d" % image_size)
        if self._general_stft():        # general STFT kernels: synthesis, then the STFT of the frames the resize keeps
            xc, flags = self._prepare(x)
            self._check_general_length(xc.shape[2])
            return self._general_image(self._general_iq(x, xc, flags, pl), image_size)
        if self._needs_grad(x, pl):     # gradients wanted: spectrogram, then torch's resize
            spec = self.forward(x) if pl is None else self._run(x, *self._prepare(x), pl)
            return torch.nn.functional.interpolate(spec.unsqueeze(1), image_size)
        xc, flags = self._prepare(x)
        noise = None
        if pl is not None:
            lam, loc, pflags, noise = pl
            flags |= pflags
        if self.assume_inputs_ready:
            flags |= _cabi.VR_FLAG_INPUTS_READY
        _, _, T, V, M = xc.shape
        N = xc.shape[0] * _cabi.views_of(flags)
        out = torch.empty((N, 1, image_size, image_size), dtype=torch.float32, device=x.device)
        if N == 0:
            return out
        with torch.cuda.device(x.device):
            stream = torch.cuda.current_stream(x.device).cuda_stream
            _set_noise(noise)
            rc = _cabi.lib().vr_forward_image_f32(xc.data_ptr(), N, T, V, M, self._src_c, self._dst_c, len(self.src),
                                                  lam.data_ptr(), loc.data_ptr(), self.n_fft, self.hop_length,
                                                  flags, image_size, out.data_ptr(), ctypes.c_void_p(stream))
        _cabi.check(rc)
        return out

    def forward_upsampled(self, x, num_pad_frames=250, sigma=3, image_size=None, radar_location=None, wavelength=None,
                          noise_std=None, noise_seed=None):
        """The data loader's temporal up-sampling fused in front of the layer: x is the RAW
        (N,3,T,V,M) batch; the result equals `self(pad_frames(x, num_pad_frames, sigma))` -- or
        `self.forward_image(pad_frames(...), image_size)` when `image_size` is given -- bit for bit,
        without the `num_pad_frames`-times larger batch ever existing in HBM (C ABI
        vr_forward_upsampled_f32; replaces reference utils.py:128-140 + layers/virtual_radar.py:79-134
        [+ models/resnet.py:24-26]).  Trainable `wavelength` / `radar_location` keep the fused path
        (vr_forward_upsampled_debug_f32 + vr_backward_upsampled_params_f32); with `image_size` the
        spectrogram is then resized by `F.interpolate`, as `forward_image` does under grad.  Gradients
        with respect to x itself go through `self(pad_frames(x, num_pad_frames, sigma))`.  `radar_location` /
        `wavelength`: per-sequence placements, and `noise_std` / `noise_seed` receiver noise, as in forward(); the noise
        is keyed by the up-sampled step, so the result equals `self(pad_frames(x, ...), noise_std=..., noise_seed=...)`."""
        self._check_input(x)
        self._check_device(x)
        pl = self._placements(x, radar_location, wavelength, noise_std, noise_seed)
        return self._upsampled(x, num_pad_frames, sigma, image_size, pl)

    def _upsampled(self, x, num_pad_frames, sigma, image_size, pl):
        """forward_upsampled after the input checks; pl: placements (_placements, _view_placements) or None."""
        lam, loc, noise = self.wavelength, self.radar_location, None
        flags = 0
        if pl is not None:
            lam, loc, flags, noise = pl
        xc = x.contiguous()
        _, _, T, V, M = xc.shape
        Nx, N = xc.shape[0], xc.shape[0] * _cabi.views_of(flags)     # raw sequences, outputs
        k = int(num_pad_frames)
        img = 0 if image_size is None else int(image_size)
        if image_size is not None and img < 1:
            raise ValueError("image_size must be positive, got %d" % img)
        if x.requires_grad and torch.is_grad_enabled():
            raise NotImplementedError("forward_upsampled has no gradient with respect to x: detach x, or differentiate "
                                      "layer(pad_frames(x, num_pad_frames, sigma)), which materialises the up-sampled batch")
        if self._general_stft():      # general STFT kernels: synthesis without the up-sampled batch, then the GEMM STFT
            if self._needs_grad(None, pl) and N > 0:
                iq = _UpsampledSynthFunction.apply(lam, loc, xc, self, k, sigma, flags, noise)
            else:
                iq = self._synth_upsampled(xc, k, sigma, lam, loc, flags, noise)[0]
            self._check_general_length(k * T)
            return self._general_image(iq, img) if img else self.stft.logmag(iq)
        if self._needs_grad(None, pl) and N > 0:
            out = _UpsampledRadarFunction.apply(lam, loc, xc, self, k, sigma, flags, noise)
            return torch.nn.functional.interpolate(out.unsqueeze(1), img) if img else out
        shape = (N, 1, img, img) if img else (N, self.n_fft, (k * T) // self.hop_length + 1)
        out = torch.empty(shape, dtype=torch.float32, device=x.device)
        if N == 0:
            return out
        L = _cabi.lib()
        nbytes = int(L.vr_upsampled_workspace_bytes(Nx, T, V, M))
        work = torch.empty(max(nbytes, 8) // 8, dtype=torch.float64, device=x.device)
        with torch.cuda.device(x.device):
            stream = torch.cuda.current_stream(x.device).cuda_stream
            # the up-sampled tensor the reference's loader builds is standard-contiguous: range rounding mode "seq"
            _set_noise(noise)
            rc = L.vr_forward_upsampled_f32(xc.data_ptr(), N, T, V, M, self._src_c, self._dst_c, len(self.src),
                                            lam.data_ptr(), loc.data_ptr(), self.n_fft, self.hop_length, flags,
                                            k, ctypes.c_float(float(sigma)), img, work.data_ptr(), nbytes,
                                            out.data_ptr(), ctypes.c_void_p(stream))
        _cabi.check(rc)
        return out

    def forward_views(self, x, radar_location, wavelength=None, image_size=None, num_pad_frames=None, sigma=3,
                      noise_std=None, noise_seed=None):
        """R radar views of every sequence in one launch from one copy of x (C ABI VR_FLAG_VIEWS(R)): a
        multistatic array, a set of viewpoints for augmentation, one scene in several bands.  x (N,3,T,V,M);
        `radar_location` float32 (R, 3), the same R placements for every sequence, or (N, R, 3); `wavelength` None (the
        module parameter), 0-d, (R,) or (N, R).  -> (N, R, n_fft, T//hop+1), or (N, R, image_size, image_size) with
        `image_size` (the forward_image fusion).  With `num_pad_frames` x is the RAW batch, up-sampled on the device as in
        forward_upsampled (its spline solved once per sequence, not once per view).  Bit for bit

            forward(x.repeat_interleave(R, 0), radar_location=loc.expand(N, R, 3).reshape(N*R, 3),
                    wavelength=lam.expand(N, R).reshape(N*R)).view(N, R, ...)

        (and likewise forward_image / forward_upsampled), without the R-times repeated batch.  Differentiable: the
        placement gradients reach the tensors passed and are the repeated route's bits; dL/dx adds the R views'
        contributions in view order, in float32, inside the kernel (deterministic; not the bits of autograd's
        repeat_interleave backward for R > 1).  As in forward_upsampled, `num_pad_frames` has no gradient with respect to
        x.  Under torch.nn.DataParallel pass full (N, R, 3) / (N, R) tensors, for the reason forward() gives.
        `noise_std` (a float or a float32 tensor that broadcasts to (N, R)) / `noise_seed`: receiver noise as in forward(),
        output n R + r keyed as output n R + r of the repeated route, so the identity above holds with the same keywords."""
        self._check_input(x)
        self._check_device(x)
        pl = self._view_placements(x, radar_location, wavelength, noise_std, noise_seed)
        if num_pad_frames is not None:
            out = self._upsampled(x, num_pad_frames, sigma, image_size, pl)
        elif image_size is not None:
            out = self._image(x, image_size, pl)
        else:
            out = self._run(x, *self._prepare(x), pl)
        return out.reshape(x.shape[0], _cabi.views_of(pl[2]), *out.shape[-2:])

    def forward_debug(self, x):
        """forward plus the intermediate complex baseband signal (N,T,2); for stage-level parity tests."""
        self._check_input(x)
        self._check_device(x)
        xc, flags = self._prepare(x)
        return self._launch(xc, flags, want_iq=True)

    def forward_host(self, x, out=None, sub_batch=0, device=None):
        """End-to-end call on HOST tensors: x (N,3,T,V,M) float32 on the CPU (pinned for full copy
        speed) -> log-spectrograms on the CPU.  Sub-batches are pipelined H2D / kernel / D2H inside
        the C library (vr_forward_host_f32)."""
        self._check_input(x)
        if x.is_cuda:
            raise ValueError("forward_host takes a CPU tensor; use forward() for CUDA tensors")
        if self._general_stft():
            raise NotImplementedError("forward_host evaluates the analytic Hann-windowed DFT only; stft.wsin/wcos are "
                                      "trained or trainable: use forward() on a CUDA tensor")
        xc, flags = self._prepare(x)
        N, _, T, V, M = xc.shape
        if out is None:
            out = torch.empty(self.output_shape(xc.shape), dtype=torch.float32, pin_memory=True)
        elif (not isinstance(out, torch.Tensor) or out.is_cuda or out.dtype != torch.float32 or not out.is_contiguous()
              or tuple(out.shape) != tuple(self.output_shape(xc.shape))):
            raise ValueError("out must be a contiguous float32 CPU tensor of shape %s" % (tuple(self.output_shape(xc.shape)),))
        if N == 0:
            return out
        dev = torch.device(device) if device is not None else self.wavelength.device
        if dev.type != "cuda":
            dev = torch.device("cuda", torch.cuda.current_device())
        lam, loc = self._host_parameters()
        with torch.cuda.device(dev):
            rc = _cabi.lib().vr_forward_host_f32(xc.data_ptr(), N, T, V, M, self._src_c, self._dst_c, len(self.src),
                                                 ctypes.c_float(lam), loc,
                                                 self.n_fft, self.hop_length, flags, out.data_ptr(), int(sub_batch))
        _cabi.check(rc)
        return out

    def _host_parameters(self):
        """Host copies of the two radar parameters for the host-buffer entry point, refreshed only when the parameters
        change (identity / version counters) -- not two device-to-host synchronisations per call."""
        key = tuple((t.data_ptr(), t._version, t.device) for t in (self.wavelength, self.radar_location))
        cached = getattr(self, "_host_params", None)
        if cached is None or cached[0] != key:
            lam = float(self.wavelength.detach().cpu())
            loc = (ctypes.c_float * 3)(*[float(v) for v in self.radar_location.detach().cpu().tolist()])
            cached = self._host_params = (key, lam, loc)
        return cached[1], cached[2]

    def extra_repr(self):
        return "bones=%d, n_fft=%d, hop_length=%d" % (len(self.src), self.n_fft, self.hop_length)
