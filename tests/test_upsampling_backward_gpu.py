"""Backward pass through the temporal up-sampling (`Dataset.pad_frames`, reference utils.py:134-140).

  * `pad_frames_adjoint` below: the adjoint of the up-sampling in numpy float64, stage by stage (the CUDA kernel's
    algorithm, vr_pad_frames.cuh); pinned on the CPU to the transpose of the dense operator that scipy itself builds
    (gaussian_filter1d(mode='reflect') + interp1d(..., 'cubic') applied to float64 unit vectors).
  * GPU: `pad_frames` is differentiable (vr_pad_frames_backward_f32), and `forward_upsampled` with trainable radar
    parameters keeps the fused path (vr_forward_upsampled_debug_f32 + vr_backward_upsampled_params_f32) instead of
    materialising the up-sampled batch.
"""
import ctypes

import numpy as np
import pytest
import torch
from scipy.interpolate import interp1d
from scipy.ndimage import gaussian_filter1d

from oracle import backward as ob
from tests import fixtures as fx


def pad_frames_adjoint(g, T, num_pad_frames, sigma):
    """dL/d(out) (..., k*T, V, M) -> dL/dx (..., T, V, M), float64: the transpose of the float64 operator
    gaussian_filter1d(sigma, axis=-3, mode='reflect') -> interp1d(linspace(0,1,T), ., 'cubic') at linspace(0,1,k*T)."""
    G = np.moveaxis(np.asarray(g, np.float64), -3, 0)
    KT = num_pad_frames * T
    assert G.shape[0] == KT
    rest = G.shape[1:]
    # evaluation: out_i = a0 + tt a1 + tt^2 a2 + tt^3 a3 of interval j (unit sample spacing)
    s = np.arange(KT, dtype=np.float64) * ((T - 1) / (KT - 1))
    j = np.minimum(s.astype(np.int64), T - 2)
    tt = (s - j).reshape((KT,) + (1,) * len(rest))
    ga = [np.zeros((T - 1,) + rest) for _ in range(4)]
    for q in range(4):
        np.add.at(ga[q], j, tt ** q * G)
    # a0 = y0, a1 = (y1 - y0) - (2 m0 + m1) / 6, a2 = m0 / 2, a3 = (m1 - m0) / 6
    gy, gM = np.zeros((T,) + rest), np.zeros((T,) + rest)
    gy[:-1] += ga[0] - ga[1]
    gy[1:] += ga[1]
    gM[:-1] += 0.5 * ga[2] - ga[1] / 3 - ga[3] / 6
    gM[1:] += (ga[3] - ga[1]) / 6
    # not-a-knot spline: 6 M1 = rhs1, 6 M(T-2) = rhs(T-2), Thomas on rows 2..T-3, M0 / M(T-1) extrapolated
    cp = np.zeros(T)
    c = 0.0
    for i in range(2, T - 2):
        c = 1.0 / (4.0 - c)
        cp[i] = c
    gM[T - 2] += 2 * gM[T - 1]
    gM[T - 3] -= gM[T - 1]
    gM[1] += 2 * gM[0]
    gM[2] -= gM[0]
    gM[0] = 0
    gM[T - 1] = 0
    for i in range(2, T - 3):
        gM[i + 1] -= cp[i] * gM[i]
    for i in range(T - 3, 1, -1):
        gM[i] *= cp[i]
        if i > 2:
            gM[i - 1] -= gM[i]
    if T >= 5:
        gM[1] -= gM[2]
        gM[T - 2] -= gM[T - 3]
    gM[1] /= 6
    gM[T - 2] /= 6
    # rhs_i = 6 (y_{i-1} - 2 y_i + y_{i+1})
    gys = gy - 12 * gM
    gys[:-1] += 6 * gM[1:]
    gys[1:] += 6 * gM[:-1]
    # reflect-padded Gaussian (scipy's _gaussian_kernel1d, radius int(4 sigma + 0.5)), transposed
    r = int(4 * float(sigma) + 0.5)
    w = np.exp(-0.5 / (float(sigma) ** 2) * np.arange(-r, r + 1) ** 2)
    w /= w.sum()
    gx = np.zeros((T,) + rest)
    t = np.arange(T)
    for off in range(-r, r + 1):
        u = np.mod(t + off, 2 * T)
        np.add.at(gx, np.where(u < T, u, 2 * T - 1 - u), w[off + r] * gys)
    return np.moveaxis(gx, 0, -3)


def _dense_operator(T, k, sigma):
    eye = np.eye(T)
    smooth = gaussian_filter1d(eye, sigma, axis=0, mode="reflect")
    return interp1d(np.linspace(0, 1, T), smooth, "cubic", axis=0)(np.linspace(0, 1, k * T))     # (k*T, T)


@pytest.mark.parametrize("sigma", [1, 3, 10])
@pytest.mark.parametrize("k", [1, 3, 10])
@pytest.mark.parametrize("T", [4, 5, 6, 13, 40])
def test_oracle_adjoint_is_the_transpose_of_scipys_operator(T, k, sigma):
    A = _dense_operator(T, k, sigma)
    g = np.random.default_rng(T * 100 + k * 10 + sigma).standard_normal((k * T, 3, 2))
    want = np.einsum("it,ivm->tvm", A, g)
    got = pad_frames_adjoint(g, T, k, sigma)
    assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max()


def test_backward_rejects_what_the_forward_rejects():
    """Argument checks that precede any device access: same return code from the forward and its backward pass."""
    from skeleton_action_recognition_b200 import _cabi
    L = _cabi.lib()
    p = ctypes.c_void_p(256)                 # never dereferenced: every case is rejected before a launch
    cases = [(None, 1, 40, 25, 2, 10, 3.0), (p, 0, 40, 25, 2, 10, 3.0), (p, 1, 3, 25, 2, 10, 3.0), (p, 1, 40, 0, 2, 10, 3.0),
             (p, 1, 40, 25, 0, 10, 3.0), (p, 1, 40, 25, 2, 0, 3.0), (p, 1, 40, 25, 2, 10, 0.0), (p, 1, 40, 25, 2, 10, -1.0),
             (p, 1, 100000, 25, 2, 100000, 3.0)]
    for src, N, T, V, M, k, sigma in cases:
        fwd = L.vr_pad_frames_f32(src, N, T, V, M, k, ctypes.c_float(sigma), p, None)
        bwd = L.vr_pad_frames_backward_f32(src, N, T, V, M, k, ctypes.c_float(sigma), p, None)
        assert fwd == bwd != 0, (src, N, T, V, M, k, sigma, fwd, bwd)
    assert L.vr_pad_frames_backward_f32(p, 1, 40, 25, 2, 10, ctypes.c_float(3.0), None, None) == _cabi.VR_ERR_ARG


# ---------------------------------------------------------------------------------------------------- GPU

def _layer(**kw):
    from skeleton_action_recognition_b200 import VirtualRadar
    return VirtualRadar(device="cuda:0", **kw).to("cuda:0")


def _raw(N, T, V, M, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(N, 3, T, V, M, generator=g) * 0.3


def _check_against_oracle(xgrad, g, T, k, sigma):
    for n in range(g.shape[0]):
        want = pad_frames_adjoint(g[n], T, k, sigma)
        got = xgrad[n].astype(np.float64)
        err = np.abs(got - want).max() / np.abs(want).max()
        assert err <= 1e-6, (n, err)


@pytest.mark.gpu
@pytest.mark.parametrize("N,T,V,M,k,sigma", [(2, 300, 25, 2, 25, 3), (1, 4, 25, 2, 10, 3), (5, 5, 7, 3, 10, 3),
                                             (1, 13, 7, 1, 3, 1), (2, 6, 5, 1, 3, 10), (1, 40, 25, 2, 1, 3)])
def test_pad_frames_backward_against_the_oracle(N, T, V, M, k, sigma):
    from skeleton_action_recognition_b200 import pad_frames
    x = _raw(N, T, V, M, T + k).cuda().requires_grad_(True)
    g = _raw(N, k * T, V, M, 7 * T + k)
    out = pad_frames(x, k, sigma)
    assert out.requires_grad
    (out * g.cuda()).sum().backward()
    _check_against_oracle(x.grad.cpu().numpy(), g.numpy(), T, k, sigma)


@pytest.mark.gpu
def test_pad_frames_backward_single_sample_out_form_and_reproducibility():
    from skeleton_action_recognition_b200 import pad_frames
    T, k, sigma = 30, 7, 3
    x = _raw(3, T, 25, 2, 11).cuda()
    g = _raw(3, k * T, 25, 2, 12).cuda()
    with torch.no_grad():
        plain = pad_frames(x, k, sigma)
    # a 4-D single sample
    x0 = x[1].clone().requires_grad_(True)
    out0 = pad_frames(x0, k, sigma)
    assert out0.shape == plain[1].shape and torch.equal(out0.detach(), plain[1])
    (out0 * g[1]).sum().backward()
    _check_against_oracle(x0.grad.unsqueeze(0).cpu().numpy(), g[1:2].cpu().numpy(), T, k, sigma)
    # the out= form carries the graph
    xo = x.clone().requires_grad_(True)
    buf = torch.empty_like(plain)
    out = pad_frames(xo, k, sigma, out=buf)
    assert out.data_ptr() == buf.data_ptr() and out.requires_grad and torch.equal(out.detach(), plain)
    (out * g).sum().backward()
    _check_against_oracle(xo.grad.cpu().numpy(), g.cpu().numpy(), T, k, sigma)
    # two runs give the same bits
    xr = x.clone().requires_grad_(True)
    (pad_frames(xr, k, sigma) * g).sum().backward()
    assert torch.equal(xr.grad, xo.grad)


@pytest.mark.gpu
def test_pad_frames_without_grad_is_unchanged():
    from skeleton_action_recognition_b200 import pad_frames
    x = _raw(2, 40, 25, 2, 13).cuda()
    out = pad_frames(x, 10, 3)
    assert out.grad_fn is None and not out.requires_grad
    xg = x.clone().requires_grad_(True)
    with torch.no_grad():
        ng = pad_frames(xg, 10, 3)
    assert ng.grad_fn is None and torch.equal(ng, out)
    assert torch.equal(pad_frames(xg, 10, 3).detach(), out)


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(wavelength=5e-3), dict(wavelength=1e-3, radar_location=[0.3, -0.2, 1.5])])
def test_gradient_wrt_the_raw_skeleton_through_pad_frames(kw):
    """dL/dx_raw of layer(pad_frames(x, 10, 3)) = oracle adjoint of the reference graph's dL/d(up-sampled x), with the
    criteria of test_gradient_wrt_the_skeleton_data (tests/test_backward_gpu.py)."""
    from skeleton_action_recognition_b200 import pad_frames
    T, k = 40, 10
    x = fx.s3_smooth(2, T=T)
    g = torch.Generator().manual_seed(8)
    go = torch.randn(2, 256, k * T // 16 + 1, generator=g)
    layer = _layer(**kw)
    xg = x.cuda().requires_grad_(True)
    up = pad_frames(xg, k, 3)
    (layer(up) * go.cuda()).sum().backward()
    got = xg.grad.cpu().numpy().astype(np.float64)
    upc = up.detach().cpu()
    for i in range(2):
        _, _, r32 = ob.autograd_grads(upc[i:i + 1], go[i:i + 1].numpy(), dtype=torch.float32, wrt_x=True, **kw)
        _, _, t64 = ob.autograd_grads(upc[i:i + 1], go[i:i + 1].numpy(), dtype=torch.float64, wrt_x=True, **kw)
        r = pad_frames_adjoint(r32[0], T, k, 3)
        t = pad_frames_adjoint(t64[0], T, k, 3)
        scale = np.linalg.norm(r) / np.sqrt(r.size)
        d_ref = np.abs(got[i] - r).max() / scale
        d_truth, ref_truth = np.abs(got[i] - t).max() / scale, np.abs(r - t).max() / scale
        print("dx_raw[%d]: gpu vs reference-f32 %.2e | vs truth-f64 %.2e (reference-f32 vs truth %.2e)" % (i, d_ref, d_truth, ref_truth))
        assert d_ref <= 2e-2 and d_truth <= 1.5 * ref_truth + 1e-3, (d_ref, d_truth, ref_truth)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [10, 250])
@pytest.mark.parametrize("image_size", [None, 64])
def test_fused_forward_with_trainable_parameters_equals_the_no_grad_output(k, image_size):
    x = fx.s3_smooth(2, T=300).cuda()
    layer = _layer(wavelength=1e-3, train_wavelength=True, train_radar_location=True)
    out = layer.forward_upsampled(x, k, 3, image_size=image_size)
    assert out.requires_grad
    with torch.no_grad():
        want = layer.forward_upsampled(x, k, 3, image_size=image_size)
    assert torch.equal(out.detach(), want)


def _fused_backward(layer, x, k, go):
    """vr_forward_upsampled_debug_f32 + vr_backward_upsampled_params_f32 through the C ABI -> (out, iq, dL/d(iq), grads)."""
    from skeleton_action_recognition_b200 import _cabi
    L = _cabi.lib()
    N, _, T, V, M = x.shape
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    nbytes = int(L.vr_upsampled_workspace_bytes(N, T, V, M))
    work = torch.empty(nbytes // 8, dtype=torch.float64, device="cuda")
    out = torch.empty(N, 256, k * T // 16 + 1, device="cuda")
    iq = torch.empty(N, k * T, 2, device="cuda")
    args = (layer._src_c, layer._dst_c, len(layer.src), layer.wavelength.data_ptr(), layer.radar_location.data_ptr(), 256, 16, 0)
    _cabi.check(L.vr_forward_upsampled_debug_f32(x.data_ptr(), N, T, V, M, *args, k, ctypes.c_float(3.0), work.data_ptr(),
                                                 nbytes, out.data_ptr(), iq.data_ptr(), stream))
    gz = torch.empty_like(iq)
    gp = torch.zeros(4, dtype=torch.float64, device="cuda")
    _cabi.check(L.vr_backward_upsampled_params_f32(work.data_ptr(), iq.data_ptr(), go.data_ptr(), N, T, V, M, *args, k,
                                                   gz.data_ptr(), gp.data_ptr(), stream))
    return out, iq, gz, gp


@pytest.mark.gpu
def test_saved_signal_and_synthesis_stage():
    """The iq the fused debug launch saves is forward_debug(pad_frames(x))[1] bit for bit, and the synthesis adjoint at the
    spline's positions equals vr_synth_adjoint_f32 on the materialised batch fed the same dL/d(iq)."""
    from skeleton_action_recognition_b200 import _cabi, pad_frames
    T, k = 300, 250
    x = fx.s3_smooth(2, T=T).cuda()
    layer = _layer(wavelength=1e-3, radar_location=[0.3, -0.2, 1.5])
    g = torch.Generator().manual_seed(9)
    go = torch.randn(2, 256, k * T // 16 + 1, generator=g).cuda()
    out, iq, gz, gp = _fused_backward(layer, x, k, go)
    up = pad_frames(x, k, 3)
    want_out, want_iq = layer.forward_debug(up)
    assert torch.equal(iq, want_iq) and torch.equal(out, want_out)
    gp_ref = torch.zeros(4, dtype=torch.float64, device="cuda")
    _cabi.check(_cabi.lib().vr_synth_adjoint_f32(up.data_ptr(), gz.data_ptr(), 2, k * T, 25, 2, layer._src_c, layer._dst_c,
                                                 len(layer.src), layer.wavelength.data_ptr(), layer.radar_location.data_ptr(),
                                                 0, gp_ref.data_ptr(), None, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    a, b = gp.cpu().numpy(), gp_ref.cpu().numpy()
    assert abs(a[0] - b[0]) <= 1e-12 * abs(b[0]), (a, b)
    assert np.abs(a[1:] - b[1:]).max() <= 1e-12 * np.abs(b[1:]).max(), (a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("kw,trainable,M", [
    (dict(wavelength=1e-3), ("wavelength", "radar_location"), 2),
    (dict(wavelength=5e-3), ("wavelength",), 2),
    (dict(wavelength=5e-3), ("radar_location",), 2),
    (dict(wavelength=1e-3, radar_location=[0.3, -0.2, 1.5]), ("wavelength", "radar_location"), 2),
    (dict(wavelength=1e-3), ("wavelength", "radar_location"), 1),
])
def test_parameter_gradients_against_the_materialising_route(kw, trainable, M):
    """Within the batch-sum tolerance of test_parameter_gradients_vs_float64_autograd: 1e-5 of the sum of the per-sequence
    gradients' magnitudes (the adjoint STFT accumulates dL/d(iq) with float32 atomics, and dL/dlambda cancels heavily)."""
    from skeleton_action_recognition_b200 import pad_frames
    T, k, N = 60, 10, 4
    x = fx.s3_smooth(N, T=T, M=M).cuda()
    g = torch.Generator().manual_seed(10)
    go = torch.randn(N, 256, k * T // 16 + 1, generator=g).cuda()
    flags = {"train_" + name: True for name in trainable}
    fused, mat = _layer(**kw, **flags), _layer(**kw, **flags)
    (fused.forward_upsampled(x, k, 3) * go).sum().backward()
    (mat(pad_frames(x, k, 3)) * go).sum().backward()
    per_seq = {name: [] for name in trainable}
    for i in range(N):
        one = _layer(**kw, **flags)
        (one(pad_frames(x[i:i + 1], k, 3)) * go[i:i + 1]).sum().backward()
        for name in trainable:
            per_seq[name].append(getattr(one, name).grad.cpu().numpy().astype(np.float64))
    for name in ("wavelength", "radar_location"):
        a, b = getattr(fused, name).grad, getattr(mat, name).grad
        if name not in trainable:
            assert a is None and b is None
            continue
        a, b = a.cpu().numpy().astype(np.float64), b.cpu().numpy().astype(np.float64)
        scale = np.abs(np.array(per_seq[name])).sum(0)
        print("%s: |fused - materialising| / sum of per-sequence magnitudes %.2e" % (name, (np.abs(a - b) / scale).max()))
        assert np.isfinite(a).all() and np.all(np.abs(a - b) <= 1e-5 * scale), (name, a, b, scale)


@pytest.mark.gpu
def test_fused_parameter_backward_does_not_materialise_the_batch():
    from skeleton_action_recognition_b200 import pad_frames
    N, T, k = 8, 300, 250
    x = fx.s3_smooth(N, T=T).cuda()
    up_bytes = N * 3 * k * T * 25 * 2 * 4
    peaks = []
    for fused in (True, False):
        layer = _layer(wavelength=1e-3, train_wavelength=True, train_radar_location=True)
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        out = layer.forward_upsampled(x, k, 3) if fused else layer(pad_frames(x, k, 3))
        out.mean().backward()
        torch.cuda.synchronize()
        peaks.append(torch.cuda.max_memory_allocated() - base)
        del out
    print("peak allocation: fused %.1f MB, materialising %.1f MB, up-sampled batch %.1f MB"
          % (peaks[0] / 1e6, peaks[1] / 1e6, up_bytes / 1e6))
    assert peaks[0] < up_bytes / 2 < peaks[1], peaks


@pytest.mark.gpu
def test_training_step_moves_the_wavelength():
    from skeleton_action_recognition_b200.models.resnet import Model
    base = torch.nn.Sequential(torch.nn.Conv2d(1, 4, 3, 2, 1), torch.nn.ReLU(), torch.nn.AdaptiveAvgPool2d(1),
                               torch.nn.Flatten(), torch.nn.Linear(4, 5))
    model = Model(num_classes=5, image_size=64, device="cuda:0", base_model=base, num_pad_frames=10).to("cuda:0")
    model.virtual_radar.wavelength.requires_grad_(True)
    opt = torch.optim.Adam([p for p in model.parameters() if p.requires_grad], lr=1e-5)
    x = fx.s3_smooth(4, T=40).cuda()
    labels = torch.tensor([0, 1, 2, 3], device="cuda")
    before = float(model.virtual_radar.wavelength.detach())
    loss = torch.nn.functional.cross_entropy(model(x), labels)
    loss.backward()
    grad = model.virtual_radar.wavelength.grad
    assert grad is not None and torch.isfinite(grad) and float(grad) != 0.0
    opt.step()
    assert float(model.virtual_radar.wavelength.detach()) != before
