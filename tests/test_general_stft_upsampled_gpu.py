"""General (trained or trainable) STFT kernels without the up-sampled batch.

  * iq-only synthesis launches (vr_synth_f32, vr_synth_upsampled_f32): bit-identical to the iq the debug launches save.
  * kept-frames STFT (vr_stft_general_frames_f32 and its backward): the columns a nearest resize reads, bit for bit the
    same as the full STFT's; gradients against the full route and float64 autograd.
  * the module: forward_upsampled / forward_image with general kernels equal the materialising compositions, with
    gradients for the kernels and the radar parameters, in a fraction of the memory.
The CPU case pins the kept-frame table to the oracle's restatement of ATen's nearest resize.
"""
import ctypes

import numpy as np
import pytest
import torch

from oracle import resize
from tests import fixtures as fx


# ---------------------------------------------------------------------------------------------------- CPU

@pytest.mark.parametrize("in_size,out_size", [(19, 256), (256, 256), (19, 64), (19, 224), (19, 300), (19, 37),
                                              (401, 256), (4688, 256), (188, 256), (512, 256), (128, 256),
                                              (10313, 256), (300, 299), (7, 1), (1251, 1000), (376, 256)])
def test_kept_frame_table_matches_the_resize_restatement(in_size, out_size):
    from skeleton_action_recognition_b200.layers.virtual_radar import kept_frame_table
    table = kept_frame_table(in_size, out_size)
    want = resize.kept_frames(in_size, out_size)
    if in_size <= out_size:           # every frame is read: the full route
        assert table is None and np.array_equal(want, np.arange(in_size))
    else:
        assert table.dtype == np.int32 and len(table) == out_size and np.array_equal(table, want)
        assert np.array_equal(table, resize.nearest_index(out_size, in_size))


# ---------------------------------------------------------------------------------------------------- GPU helpers

def _layer(**kw):
    from skeleton_action_recognition_b200 import VirtualRadar
    return VirtualRadar(device="cuda:0", **kw).to("cuda:0")


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _synth(layer, xc, flags):
    from skeleton_action_recognition_b200 import _cabi
    N, _, T, V, M = xc.shape
    iq = torch.full((N, T, 2), float("nan"), device="cuda")
    _cabi.check(_cabi.lib().vr_synth_f32(xc.data_ptr(), N, T, V, M, layer._src_c, layer._dst_c, len(layer.src),
                                         layer.wavelength.data_ptr(), layer.radar_location.data_ptr(), flags,
                                         iq.data_ptr(), _stream()))
    return iq


def _debug(layer, xc, flags):
    from skeleton_action_recognition_b200 import _cabi
    N, _, T, V, M = xc.shape
    out = torch.empty(N, 256, T // 16 + 1, device="cuda")
    iq = torch.full((N, T, 2), float("nan"), device="cuda")
    _cabi.check(_cabi.lib().vr_forward_debug_f32(xc.data_ptr(), N, T, V, M, layer._src_c, layer._dst_c, len(layer.src),
                                                 layer.wavelength.data_ptr(), layer.radar_location.data_ptr(), 256, 16,
                                                 flags, out.data_ptr(), iq.data_ptr(), _stream()))
    return iq


def _synth_upsampled(layer, x, k, sigma, debug):
    from skeleton_action_recognition_b200 import _cabi
    L = _cabi.lib()
    N, _, T, V, M = x.shape
    nbytes = int(L.vr_upsampled_workspace_bytes(N, T, V, M))
    work = torch.empty(nbytes // 8, dtype=torch.float64, device="cuda")
    iq = torch.full((N, k * T, 2), float("nan"), device="cuda")
    args = (x.data_ptr(), N, T, V, M, layer._src_c, layer._dst_c, len(layer.src), layer.wavelength.data_ptr(),
            layer.radar_location.data_ptr())
    if debug:
        out = torch.empty(N, 256, k * T // 16 + 1, device="cuda")
        rc = L.vr_forward_upsampled_debug_f32(*args, 256, 16, 0, k, ctypes.c_float(sigma), work.data_ptr(), nbytes,
                                              out.data_ptr(), iq.data_ptr(), _stream())
    else:
        rc = L.vr_synth_upsampled_f32(*args, 0, k, ctypes.c_float(sigma), work.data_ptr(), nbytes, iq.data_ptr(), _stream())
    _cabi.check(rc)
    return iq


def _chain_edges(E):
    return [(i, i + 1) for i in range(E)]


def _kernels(n_fft, hop, perturb, seed=0):
    from skeleton_action_recognition_b200.layers.virtual_radar import _STFTKernels
    k = _STFTKernels(n_fft, hop, True, "cuda:0")
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        k.wsin.add_((perturb * torch.randn(k.wsin.shape, generator=g)).cuda())
        k.wcos.add_((perturb * torch.randn(k.wcos.shape, generator=g)).cuda())
    return k


def _perturb(layer, seed=5, eps=0.02):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        layer.stft.wsin.add_((eps * torch.randn(layer.stft.wsin.shape, generator=g)).cuda())
        layer.stft.wcos.add_((eps * torch.randn(layer.stft.wcos.shape, generator=g)).cuda())
    return layer


# ---------------------------------------------------------------------------------------------------- 1. vr_synth_f32

@pytest.mark.gpu
@pytest.mark.parametrize("N,T,V,M,fma,E", [
    (1, 300, 25, 2, False, None), (257, 300, 25, 2, False, None), (2000, 300, 25, 2, True, None),
    (3, 300, 25, 1, False, None), (3, 300, 25, 3, True, None),
    (2, 301, 7, 3, False, 6),                        # T*V*M = 6321: no TMA loads, ragged planes
    (4, 129, 25, 2, True, None), (2, 75000, 25, 2, False, None), (2, 75000, 25, 1, True, None),
    (3, 300, 129, 1, False, 128),                    # 128 bones, 32 per lane group
])
def test_synth_iq_equals_the_debug_launch(N, T, V, M, fma, E):
    from skeleton_action_recognition_b200 import _cabi
    kw = dict(wavelength=1e-3, radar_location=[0.3, -0.2, 1.5])
    layer = _layer(edges=_chain_edges(E), **kw) if E else _layer(**kw)
    g = torch.Generator().manual_seed(N + T + V + M)
    x = (torch.randn(N, 3, T, V, M, generator=g) * 0.3).cuda()
    flags = _cabi.VR_FLAG_RANGE_FMA if fma else 0
    got = _synth(layer, x, flags)
    want = _debug(layer, x, flags)
    assert torch.equal(got, want)
    # the module's no-grad synthesis is the same launch
    assert torch.equal(layer._synth(x, flags), want)


@pytest.mark.gpu
def test_synth_needs_no_stft_length():
    """T <= n_fft/2 is fine for the synthesis alone: it equals the first samples of a longer sequence's synthesis."""
    layer = _layer(wavelength=1e-3)
    x = fx.s3_smooth(2, T=300).cuda()
    full = _synth(layer, x, 0)
    for T in (1, 31, 32, 33, 100):
        assert torch.equal(_synth(layer, x[:, :, :T].contiguous(), 0), full[:, :T]), T


# ---------------------------------------------------------------------------------------------------- 2. up-sampled

@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 10, 250])
@pytest.mark.parametrize("sigma", [1, 3])
@pytest.mark.parametrize("T", [4, 5, 40, 300])
def test_synth_upsampled_iq_equals_the_debug_launches(k, sigma, T):
    from skeleton_action_recognition_b200 import pad_frames
    layer = _layer(wavelength=1e-3, radar_location=[0.3, -0.2, 1.5])
    x = fx.s3_smooth(2, T=T).cuda() if T >= 40 else (torch.randn(2, 3, T, 25, 2, generator=torch.Generator().manual_seed(T)) * 0.3).cuda()
    got = _synth_upsampled(layer, x, k, float(sigma), debug=False)
    up = pad_frames(x, k, sigma)
    if k * T > 128:
        assert torch.equal(got, _synth_upsampled(layer, x, k, float(sigma), debug=True))
        assert torch.equal(got, layer.forward_debug(up)[1])
    else:
        assert torch.equal(got, _synth(layer, up, 0))


# ---------------------------------------------------------------------------------------------------- 3. kept-frames forward

def _tables(F, n_fft, hop):
    step = -(-n_fft // hop)                                        # frames this far apart do not overlap
    mid = F // 2
    return {
        "overlapping": sorted({0, F - 1} | set(range(max(mid - 3, 0), min(mid + 4, F)))),
        "disjoint": list(range(1, F - 1, step + 1)) or [F // 2],
        "nearest": resize.kept_frames(F, max(F // 3, 1)).tolist(),
    }


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft", [16, 64, 256, 1024])
@pytest.mark.parametrize("hop", [8, 13, 16, 100])
def test_kept_frames_forward_equals_the_columns_of_the_full_stft(n_fft, hop):
    T = n_fft + 37 * hop + 5
    F = T // hop + 1
    N = 3
    g = torch.Generator().manual_seed(n_fft * hop)
    iq = torch.randn(N, T, 2, generator=g).cuda()
    k = _kernels(n_fft, hop, 0.02, seed=hop)
    with torch.no_grad():
        full = k.logmag(iq)
        for name, table in _tables(F, n_fft, hop).items():
            fr = torch.tensor(table, dtype=torch.int32, device="cuda")
            got = k.logmag(iq, fr)
            assert got.shape == (N, n_fft, len(table)), name
            assert torch.equal(got, full[:, :, fr.long()]), (name, table)


# ---------------------------------------------------------------------------------------------------- 5. kept-frames backward

@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop,T,N,S", [(256, 16, 5000, 3, 256), (128, 16, 1200, 2, 40), (64, 13, 700, 3, 17),
                                             (16, 8, 300, 2, 7)])
def test_kept_frames_backward(n_fft, hop, T, N, S):
    interp = torch.nn.functional.interpolate
    F = T // hop + 1
    assert F > S
    g = torch.Generator().manual_seed(n_fft + S)
    iq = torch.randn(N, T, 2, generator=g)
    go = torch.randn(N, 1, S, S, generator=g).cuda()
    frames = torch.from_numpy(resize.kept_frames(F, S).astype(np.int32)).cuda()
    # kept route and full route, same kernels
    kk, kf = _kernels(n_fft, hop, 0.02, seed=1), _kernels(n_fft, hop, 0.02, seed=1)
    xk, xf = iq.cuda().requires_grad_(True), iq.cuda().requires_grad_(True)
    spec_k = kk.logmag(xk, frames)
    yk = interp(spec_k.unsqueeze(1), S)
    spec_f = kf.logmag(xf)
    assert torch.equal(yk, interp(spec_f.unsqueeze(1), S))
    g_kept, = torch.autograd.grad((yk * go).sum(), spec_k)
    # the full route fed F.interpolate's backward, column c's gradient going to the frame the forward read for c.  (ATen's
    # CUDA nearest backward maps columns to frames with its own float rounding, which at (F, S) = (76, 40) sends column 30's
    # gradient to frame 56 although the forward read frame 57: interpolating the full spectrogram under autograd then
    # differentiates a different function than it evaluates.  The compact spectrogram is resized with column scale 1.)
    g_full = torch.zeros_like(spec_f)
    g_full[:, :, frames.long()] = g_kept
    spec_k.backward(g_kept)
    spec_f.backward(g_full)
    # dL/d(iq): dC of a frame the resize does not read is zero, the frame-gradient GEMM is row by row, and the kept fold sums
    # the same non-zero terms in the same order -- so the two are equal
    assert torch.equal(xk.grad, xf.grad)
    # float64 truth of the same graph, and the float32 torch restatement as the yardstick (as test_stft_general_gpu.py)
    k64 = _kernels(n_fft, hop, 0.0).double().cpu()
    kl = _kernels(n_fft, hop, 0.0)
    with torch.no_grad():
        for dst in (k64, kl):
            dst.wsin.copy_(kk.wsin.detach().to(dst.wsin))
            dst.wcos.copy_(kk.wcos.detach().to(dst.wcos))
    x64 = iq.double().requires_grad_(True)
    (interp(k64._logmag_torch(x64).unsqueeze(1), S) * go.cpu().double()).sum().backward()
    xl = iq.cuda().requires_grad_(True)
    (interp(kl._logmag_torch(xl).unsqueeze(1), S) * go).sum().backward()
    for name, a, b, c in (("iq", xk.grad, x64.grad, xl.grad), ("wsin", kk.wsin.grad, k64.wsin.grad, kl.wsin.grad),
                          ("wcos", kk.wcos.grad, k64.wcos.grad, kl.wcos.grad)):
        a, c = a.cpu().double(), c.cpu().double()
        scale = b.square().mean().sqrt()
        err, err_lib = (a - b).abs().max() / scale, (c - b).abs().max() / scale
        med, med_lib = (a - b).abs().median() / scale, (c - b).abs().median() / scale
        print("%s: kept max %.2e median %.2e | library f32 max %.2e median %.2e" % (name, err, med, err_lib, med_lib))
        assert err < max(3 * err_lib, 2e-4) and med < max(3 * med_lib, 2e-6), (name, float(err), float(err_lib), float(med), float(med_lib))
    # the kernel gradients of the two routes differ only in the order of the float sums over frames
    for a, b in ((kk.wsin.grad, kf.wsin.grad), (kk.wcos.grad, kf.wcos.grad)):
        assert float((a - b).abs().max() / b.square().mean().sqrt()) < 1e-4


# ---------------------------------------------------------------------------------------------------- 4. module, bit-exact

_GENERAL = {
    "perturbed-frozen": lambda: _perturb(_layer(wavelength=1e-3)),
    "trainable": lambda: _perturb(_layer(wavelength=1e-3, train_stft_kernel=True)),
    "nfft128": lambda: _layer(wavelength=1e-3, n_fft=128),
    "nfft512-trainable": lambda: _perturb(_layer(wavelength=1e-3, n_fft=512, hop_length=32, train_stft_kernel=True)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("config", sorted(_GENERAL))
@pytest.mark.parametrize("k,T,S", [(10, 40, 16), (250, 300, 256), (10, 300, 64)])
@pytest.mark.parametrize("grad", [False, True])
def test_module_forward_upsampled_equals_the_materialising_composition(config, k, T, S, grad):
    from skeleton_action_recognition_b200 import pad_frames
    layer = _GENERAL[config]()
    assert layer._general_stft()
    x = fx.s3_smooth(2, T=T).cuda()
    with torch.set_grad_enabled(grad):
        up = pad_frames(x, k, 3)
        spec = layer.forward_upsampled(x, k, 3)
        img = layer.forward_upsampled(x, k, 3, image_size=S)
        want_spec = layer(up)
        want_img = layer.forward_image(up, S)
        want_interp = torch.nn.functional.interpolate(want_spec.unsqueeze(1), S)
    assert spec.requires_grad == (grad and layer.stft.wsin.requires_grad)
    assert torch.equal(spec, want_spec) and torch.equal(img, want_img) and torch.equal(img, want_interp)


@pytest.mark.gpu
@pytest.mark.parametrize("T,S", [(300, 64), (300, 8), (5000, 256)])
def test_forward_image_with_trained_kernels_equals_interpolate(T, S):
    layer = _perturb(_layer(wavelength=1e-3, train_stft_kernel=True, train_wavelength=True))
    x = fx.s3_smooth(2, T=T).cuda()
    got = layer.forward_image(x, S)
    want = torch.nn.functional.interpolate(layer(x).unsqueeze(1), S)
    assert got.requires_grad and torch.equal(got, want)
    with torch.no_grad():
        assert torch.equal(layer.forward_image(x, S), want)


# ---------------------------------------------------------------------------------------------------- 6. module gradients

@pytest.mark.gpu
@pytest.mark.parametrize("S", [None, 16])
@pytest.mark.parametrize("kw", [dict(wavelength=1e-3), dict(wavelength=1e-3, radar_location=[0.3, -0.2, 1.5])])
def test_module_gradients_against_the_materialising_composition(S, kw):
    from skeleton_action_recognition_b200 import pad_frames
    interp = torch.nn.functional.interpolate
    T, k, N = 60, 10, 4
    x = fx.s3_smooth(N, T=T).cuda()
    flags = dict(train_stft_kernel=True, train_wavelength=True, train_radar_location=True)
    F = k * T // 16 + 1
    go = torch.randn((N, 1, S, S) if S else (N, 256, F), generator=torch.Generator().manual_seed(3)).cuda()

    def run(layer, xx, gg, fused):
        if fused:
            out = layer.forward_upsampled(xx, k, 3, image_size=S)
        else:
            out = layer(pad_frames(xx, k, 3))
            out = interp(out.unsqueeze(1), S) if S else out
        (out * gg).sum().backward()

    fused, mat = _perturb(_layer(**kw, **flags)), _perturb(_layer(**kw, **flags))
    run(fused, x, go, True)
    run(mat, x, go, False)
    per_seq = {"wavelength": [], "radar_location": []}
    for i in range(N):
        one = _perturb(_layer(**kw, **flags))
        run(one, x[i:i + 1], go[i:i + 1], False)
        for name in per_seq:
            per_seq[name].append(getattr(one, name).grad.cpu().numpy().astype(np.float64))
    for name in per_seq:
        a = getattr(fused, name).grad.cpu().numpy().astype(np.float64)
        b = getattr(mat, name).grad.cpu().numpy().astype(np.float64)
        scale = np.abs(np.array(per_seq[name])).sum(0)
        print("%s: |new - materialising| / sum of per-sequence magnitudes %.2e" % (name, (np.abs(a - b) / scale).max()))
        assert np.isfinite(a).all() and np.all(np.abs(a - b) <= 1e-5 * scale), (name, a, b, scale)
    for name in ("wsin", "wcos"):
        a, b = getattr(fused.stft, name).grad.double(), getattr(mat.stft, name).grad.double()
        rms = b.square().mean().sqrt()
        err, med = float((a - b).abs().max() / rms), float((a - b).abs().median() / rms)
        print("%s: |new - materialising| max %.2e median %.2e of the rms" % (name, err, med))
        assert err < 2e-4 and med < 2e-6, (name, err, med)


# ---------------------------------------------------------------------------------------------------- 7. memory

@pytest.mark.gpu
def test_general_route_does_not_materialise_the_batch():
    N, T, k, S = 8, 300, 250, 256
    x = fx.s3_smooth(N, T=T).cuda()
    up_bytes = N * 3 * k * T * 25 * 2 * 4
    layer = _layer(wavelength=1e-3, train_stft_kernel=True, train_wavelength=True, train_radar_location=True)
    layer.forward_upsampled(x[:1], k, 3, image_size=S).mean().backward()      # kept-frame table and library warm
    layer.zero_grad(set_to_none=True)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    out = layer.forward_upsampled(x, k, 3, image_size=S)
    out.mean().backward()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    print("peak allocation %.1f MB, up-sampled batch %.1f MB" % (peak / 1e6, up_bytes / 1e6))
    assert peak < up_bytes / 4, (peak, up_bytes)


# ---------------------------------------------------------------------------------------------------- 8. edge cases

@pytest.mark.gpu
def test_no_grad_saves_nothing():
    layer = _layer(wavelength=1e-3, train_stft_kernel=True, train_wavelength=True)
    x = fx.s3_smooth(2, T=300).cuda()
    with torch.no_grad():
        layer.forward_upsampled(x, 250, 3, image_size=256)
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        out = layer.forward_upsampled(x, 250, 3, image_size=256)
        torch.cuda.synchronize()
        kept = torch.cuda.memory_allocated() - base
    assert out.grad_fn is None and not out.requires_grad
    assert kept <= out.numel() * 4 + 512, kept


@pytest.mark.gpu
@pytest.mark.parametrize("S", [None, 256])
def test_eval_after_an_optimizer_step_sees_the_new_kernels(S):
    from skeleton_action_recognition_b200 import pad_frames
    layer = _layer(wavelength=1e-3, train_stft_kernel=True)
    x = fx.s3_smooth(2, T=300).cuda()
    with torch.no_grad():
        before = layer.forward_upsampled(x, 250, 3, image_size=S)
    opt = torch.optim.SGD(layer.parameters(), lr=1e-2)
    layer.forward_upsampled(x, 250, 3, image_size=S).square().mean().backward()
    opt.step()
    with torch.no_grad():
        after = layer.forward_upsampled(x, 250, 3, image_size=S)
        up = pad_frames(x, 250, 3)
        want = layer.forward_image(up, S) if S else layer(up)
    assert not torch.equal(after, before) and torch.equal(after, want)


@pytest.mark.gpu
def test_edge_cases():
    from skeleton_action_recognition_b200 import pad_frames
    layer = _layer(wavelength=1e-3, train_stft_kernel=True, train_wavelength=True)
    x = fx.s3_smooth(2, T=40).cuda()
    with pytest.raises(NotImplementedError):
        layer.forward_upsampled(x.clone().requires_grad_(True), 10, 3)
    empty = torch.empty(0, 3, 40, 25, 2, device="cuda")
    assert layer.forward_upsampled(empty, 10, 3).shape == (0, 256, 10 * 40 // 16 + 1)
    assert layer.forward_upsampled(empty, 10, 3, image_size=16).shape == (0, 1, 16, 16)
    with torch.no_grad():
        assert layer.forward_upsampled(empty, 10, 3).shape == (0, 256, 10 * 40 // 16 + 1)
    # too short for the STFT's reflect padding: the same error as the materialising composition
    short = x[:, :, :4].contiguous()
    with pytest.raises(ValueError) as new:
        layer.forward_upsampled(short, 10, 3)
    with pytest.raises(ValueError) as old:
        layer(pad_frames(short, 10, 3))
    assert str(new.value) == str(old.value)
    with pytest.raises(ValueError) as new_img:
        layer.forward_upsampled(short, 10, 3, image_size=16)
    assert str(new_img.value) == str(old.value)


# ---------------------------------------------------------------------------------------------------- 9. training step

@pytest.mark.gpu
def test_training_step_moves_the_stft_kernels():
    from skeleton_action_recognition_b200.models.resnet import Model
    base = torch.nn.Sequential(torch.nn.Conv2d(1, 4, 3, 2, 1), torch.nn.ReLU(), torch.nn.AdaptiveAvgPool2d(1),
                               torch.nn.Flatten(), torch.nn.Linear(4, 5))
    model = Model(num_classes=5, image_size=64, device="cuda:0", base_model=base, num_pad_frames=10).to("cuda:0")
    vr = model.virtual_radar
    vr.stft.wsin.requires_grad_(True)
    vr.stft.wcos.requires_grad_(True)
    opt = torch.optim.Adam([p for p in model.parameters() if p.requires_grad], lr=1e-3)
    x = fx.s3_smooth(4, T=40).cuda()
    labels = torch.tensor([0, 1, 2, 3], device="cuda")
    before = vr.stft.wsin.detach().clone()
    loss = torch.nn.functional.cross_entropy(model(x), labels)
    assert torch.isfinite(loss)
    loss.backward()
    assert torch.isfinite(vr.stft.wsin.grad).all() and float(vr.stft.wsin.grad.abs().max()) > 0
    opt.step()
    assert not torch.equal(vr.stft.wsin.detach(), before)
