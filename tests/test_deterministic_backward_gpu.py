"""Bitwise-reproducible gradients.  The backward entry points return the same dL/d(iq), dL/dx and radar-parameter gradients
when called again on the same inputs -- serially, on two streams at once, or replayed from a CUDA graph -- and the
per-sequence gradients (dL/d(iq), dL/dx) of a sequence do not depend on the rest of the batch.  The owner-form adjoint STFT and the fixed-order
parameter reduction stay within the oracle tolerances of tests/test_backward_property_gpu.py, and a few SGD steps of a
module under torch.use_deterministic_algorithms(True) end in the same parameters every time."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import backward as ob
from tests.test_backward_property_gpu import (OFF_AXIS, _layer, _positions, _stream, backward_gpu, check_module,
                                              check_stft_adjoint, synth_gpu)

pytestmark = pytest.mark.gpu

SMALL_EDGES = [(0, 1), (1, 2), (2, 3), (1, 4), (4, 5), (0, 6)]


def _ntu_edges():
    from skeleton_action_recognition_b200 import edges
    return [tuple(e) for e in edges]


def _case(N, T, V, M, edges, hop, seed):
    """x on the GPU, the forward's saved iq and a random dL/d(out)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(N, 3, T, V, M, device="cuda", generator=g) * 0.4
    layer = _layer(edges, 1e-3, OFF_AXIS, hop)
    _, iq = layer.forward_debug(x)
    go = torch.randn(N, 256, T // hop + 1, device="cuda", generator=g)
    return x, iq, go


def _same(a, b):
    """bit equality (NaN-safe)"""
    return a.shape == b.shape and torch.equal(a.reshape(-1).view(torch.int8), b.reshape(-1).view(torch.int8))


# ---- the default-kernel backward (vr_backward_f32) ------------------------------------------------------------------------------
@pytest.mark.parametrize("N,T,ntu", [(64, 300, True), (4096, 300, True), (4, 75000, True), (300, 2100, False)])
def test_backward_repeats_bit_for_bit(N, T, ntu):
    """NTU shapes at the batch sizes where the old overlap-add and parameter atomics contended, a 75 000-step sequence
    (several adjoint segments per sequence), and a batch that makes the synthesis grid loop."""
    edges = _ntu_edges() if ntu else [(0, 1), (1, 2), (2, 3), (3, 4), (1, 5), (5, 6), (6, 7), (0, 8), (8, 9), (9, 10)]
    V, M = (25, 2) if ntu else (11, 3)
    x, iq, go = _case(N, T, V, M, edges, 16, 11)
    want_x = N * T <= 4096 * 300
    first = backward_gpu(x, iq, go, edges, 1e-3, OFF_AXIS, 16, 0, want_x=want_x)
    second = backward_gpu(x, iq, go, edges, 1e-3, OFF_AXIS, 16, 0, want_x=want_x)
    for a, b, name in zip(first, second, ("gz", "grad_params", "grad_x")):
        if a is not None:
            assert _same(a, b), name
    gp, gx = synth_gpu(x, first[0], edges, 1e-3, OFF_AXIS, 0, want_x=want_x)
    assert _same(gp, first[1])
    if want_x:
        assert _same(gx, first[2])


@pytest.mark.parametrize("N,T,hop", [(64, 300, 16), (300, 2100, 16), (4, 75000, 16), (24, 1000, 300)])
def test_batch_slice_invariance(N, T, hop):
    """dL/d(iq) and dL/dx of sequence n inside the batch equal those of x[n:n+1] alone.  At T = 2100 and 75 000 the batch
    and the single sequence get different segment cuts (vr_plan_adjoint_stft); the sums do not change."""
    from skeleton_action_recognition_b200 import _cabi
    edges = SMALL_EDGES
    x, iq, go = _case(N, T, 7, 3, edges, hop, 21)
    if T == 2100:
        assert _cabi.plan_adjoint_stft(N, T, hop)[0]["segments"] != _cabi.plan_adjoint_stft(1, T, hop)[0]["segments"]
    gz, _, gx = backward_gpu(x, iq, go, edges, 1e-3, OFF_AXIS, hop, 0)
    for n in sorted({0, 1, N // 2, N - 1}):
        gz1, _, gx1 = backward_gpu(x[n:n + 1].contiguous(), iq[n:n + 1].contiguous(), go[n:n + 1].contiguous(), edges,
                                   1e-3, OFF_AXIS, hop, 0)
        assert _same(gz1[0], gz[n]), n
        assert _same(gx1[0], gx[n]), n


def test_concurrent_streams_and_graph_replay():
    """Two backward calls issued at once on two streams, and a backward captured in a CUDA graph and replayed, equal the
    serial result: each launch has its own slot of the parameter partials."""
    edges = _ntu_edges()
    x, iq, go = _case(512, 300, 25, 2, edges, 16, 31)
    ref = backward_gpu(x, iq, go, edges, 1e-3, OFF_AXIS, 16, 0)
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    outs = [None, None]
    for _ in range(3):
        for i, s in enumerate(streams):
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                outs[i] = backward_gpu(x, iq, go, edges, 1e-3, OFF_AXIS, 16, 0)
        torch.cuda.synchronize()
        for o in outs:
            for a, b in zip(o, ref):
                assert _same(a, b)
    # graph: the parameter accumulator is zeroed inside the graph (the entry point adds to it)
    from skeleton_action_recognition_b200 import _cabi
    from tests.test_backward_property_gpu import _params
    N, _, T, V, M = x.shape
    lam_t, loc_t = _params(1e-3, OFF_AXIS)
    gz = torch.empty(N, T, 2, device="cuda")
    gp = torch.zeros(4, dtype=torch.float64, device="cuda")
    gx = torch.empty_like(x)
    src, dst = map(list, zip(*edges))
    src_c, dst_c = _cabi.i32_array(src), _cabi.i32_array(dst)

    def call():
        gp.zero_()
        _cabi.check(_cabi.lib().vr_backward_f32(x.data_ptr(), iq.data_ptr(), go.data_ptr(), N, T, V, M, src_c, dst_c,
                                                len(src), lam_t.data_ptr(), loc_t.data_ptr(), 256, 16, 0, gz.data_ptr(),
                                                gp.data_ptr(), gx.data_ptr(), _stream()))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        call()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        call()
    for _ in range(3):
        gz.fill_(float("nan"))
        gx.fill_(float("nan"))
        graph.replay()
        torch.cuda.synchronize()
        assert _same(gz, ref[0]) and _same(gp, ref[1]) and _same(gx, ref[2])


# ---- the up-sampled parameter backward (vr_backward_upsampled_params_f32) -------------------------------------------------------
def test_upsampled_backward_repeats_bit_for_bit():
    from tests.test_upsampling_backward_gpu import _fused_backward
    from skeleton_action_recognition_b200 import VirtualRadar
    import tests.fixtures as fx
    k, N, T = 250, 8, 300
    x = fx.s3_smooth(N, T=T).cuda()
    layer = VirtualRadar(wavelength=1e-3, radar_location=list(OFF_AXIS), device="cuda:0").to("cuda:0")
    go = torch.randn(N, 256, k * T // 16 + 1, generator=torch.Generator().manual_seed(41)).cuda()
    _, _, gz1, gp1 = _fused_backward(layer, x, k, go)
    _, _, gz2, gp2 = _fused_backward(layer, x, k, go)
    assert _same(gz1, gz2) and _same(gp1, gp2)
    _, _, gz3, _ = _fused_backward(layer, x[2:3].contiguous(), k, go[2:3].contiguous())
    assert _same(gz3[0], gz1[2])


# ---- the general-kernel STFT backward (vr_stft_general*_backward_f32) -----------------------------------------------------------
def _general(n_fft, N, T, kept, seed):
    from skeleton_action_recognition_b200 import VirtualRadar
    layer = VirtualRadar(train_stft_kernel=True, n_fft=n_fft, device="cuda:0").to("cuda:0")
    g = torch.Generator(device="cuda").manual_seed(seed)
    iq = torch.randn(N, T, 2, device="cuda", generator=g)
    F = T // 16 + 1
    frames = None
    if kept:
        frames = torch.arange(0, F, 3, dtype=torch.int32, device="cuda")
    ncols = F if frames is None else frames.numel()
    go = torch.randn(N, n_fft, ncols, device="cuda", generator=g)

    def run(sl=slice(None)):
        for p in (layer.stft.wsin, layer.stft.wcos):
            p.grad = None
        i = iq[sl].clone().requires_grad_(True)
        (layer.stft.logmag(i, frames) * go[sl]).sum().backward()
        return i.grad, layer.stft.wsin.grad.clone(), layer.stft.wcos.grad.clone()
    return run


@pytest.mark.parametrize("kept", [False, True], ids=["full", "kept"])
@pytest.mark.parametrize("n_fft", [64, 128, 256, 512, 1024])
def test_general_stft_backward_repeats_bit_for_bit(n_fft, kept):
    """All three gradients of the general STFT on both routes, at batches where the kernel-gradient reduction is split
    (N * F > 256 frames: up to 148 slices at n_fft = 64, 9 at 256, 2 at 512; n_fft = 1024 has 256 output tiles, one slice):
    repeat equality, and dL/d(iq) of the last sequence equals that of the sequence alone."""
    T = 300 if n_fft <= 256 else 1300                           # T > n_fft / 2
    N = 512 if n_fft <= 256 else 128
    run = _general(n_fft, N, T, kept, 51)
    a, b = run(), run()
    for u, v, name in zip(a, b, ("grad_iq", "grad_wsin", "grad_wcos")):
        assert _same(u, v), name
    assert _same(run(slice(N - 1, N))[0][0], a[0][N - 1])


def test_ntu_kernel_gradients_repeat_bit_for_bit():
    """train_stft_kernel=True through the module at NTU shape, N = 4096 (77 824 frames, 9 slices at n_fft = 256): the kernel
    gradients of two backward passes are equal bit for bit, also under torch.use_deterministic_algorithms(True)."""
    from skeleton_action_recognition_b200 import VirtualRadar
    layer = VirtualRadar(wavelength=1e-3, train_stft_kernel=True, device="cuda:0").to("cuda:0")
    x = torch.randn(4096, 3, 300, 25, 2, device="cuda", generator=torch.Generator(device="cuda").manual_seed(81)) * 0.4
    before = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        grads = []
        for _ in range(2):
            layer.zero_grad()
            layer(x).square().mean().backward()
            grads.append((layer.stft.wsin.grad.clone(), layer.stft.wcos.grad.clone()))
    finally:
        torch.use_deterministic_algorithms(before)
    assert _same(grads[0][0], grads[1][0]) and _same(grads[0][1], grads[1][1])
    assert float(grads[0][0].abs().max()) > 0


# ---- accuracy of the new sums ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T", [129, 1000, 2100])
@pytest.mark.parametrize("hop", [8, 16, 100, 300])
def test_oracle_accuracy(T, hop):
    """The owner-form dL/d(iq) and the reduced parameter gradients within the oracle checks of the property tests; with
    hop > n_fft, the samples no frame covers are exactly 0."""
    x = _positions((2, 3, T, 7, 3), 60 + hop)
    check_module("T=%d hop=%d" % (T, hop), x, SMALL_EDGES, 1e-3, OFF_AXIS, hop, 61 + T)
    if hop > 256:
        xc = x.cuda().contiguous()
        layer = _layer(SMALL_EDGES, 1e-3, OFF_AXIS, hop)
        _, iq = layer.forward_debug(xc)
        go = torch.randn(2, 256, T // hop + 1, generator=torch.Generator().manual_seed(62)).cuda()
        gz, _, _ = backward_gpu(xc, iq, go, SMALL_EDGES, 1e-3, OFF_AXIS, hop, 0, want_x=False)
        covered = np.zeros(T, bool)
        for f in range(T // hop + 1):
            covered[ob._reflect(f * hop - 128 + np.arange(256), T)] = True
        assert T < 1000 or (~covered).sum() > 0                 # T = 129: frame 0 covers everything
        assert (gz.cpu().numpy()[:, ~covered] == 0).all()
        assert (np.abs(gz.cpu().numpy()[:, covered]).sum(-1) > 0).any()


def test_grid_stride_sizes_repeat_and_match_the_oracle():
    """The sizes of test_grid_stride_wrap (the synthesis grid loops): repeat equality, and dL/d(iq) of three sequences
    against the oracle."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    T, hop, V, M = 2100, 16, 11, 3
    N = 2 * (16 * 128 * sms + T - 1) // T + 1
    edges = [(0, 1), (1, 2), (2, 3), (3, 4), (1, 5), (5, 6), (6, 7), (0, 8), (8, 9), (9, 10), (5, 5 + 2), (2, 9)]
    x, iq, go = _case(N, T, V, M, edges, hop, 61)
    a = backward_gpu(x, iq, go, edges, 1e-3, OFF_AXIS, hop, 0)
    b = backward_gpu(x, iq, go, edges, 1e-3, OFF_AXIS, hop, 0)
    for u, v in zip(a, b):
        assert _same(u, v)
    for n in (0, N // 2, N - 1):
        check_stft_adjoint("grid-stride n=%d" % n, a[0][n:n + 1], iq[n:n + 1], go[n:n + 1], hop)


# ---- module level: SGD under torch.use_deterministic_algorithms(True) -----------------------------------------------------------
def _sgd_run(case, steps=3):
    """Three SGD steps of a VirtualRadar and a small head from a fixed state and batch -> every parameter after them."""
    from skeleton_action_recognition_b200 import VirtualRadar
    train_radar = case in ("radar", "ups_radar")
    layer = VirtualRadar(wavelength=1e-3, radar_location=[0.3, -0.2, 1.5], train_wavelength=train_radar,
                         train_radar_location=train_radar, train_stft_kernel=not train_radar, device="cuda:0").to("cuda:0")
    g = torch.Generator(device="cuda").manual_seed(71)
    # kernel-gradient cases above 256 frames, so that their reduction is split: 64 x 19 frames, 8 x 38 up-sampled ones
    N, T = {"radar": (6, 300), "stft": (64, 300), "ups_radar": (3, 60), "ups_stft": (8, 60)}[case]
    x = (torch.randn(N, 3, T, 25, 2, device="cuda", generator=g) * 0.4).requires_grad_(case == "radar")
    target = torch.randn(N, device="cuda", generator=g)
    head = torch.nn.Parameter(torch.linspace(-1.0, 1.0, 256, device="cuda"))
    groups = [{"params": [head], "lr": 1e-3}]
    if train_radar:
        groups += [{"params": [layer.wavelength], "lr": 1e-14}, {"params": [layer.radar_location], "lr": 1e-8}]
    else:
        groups += [{"params": [layer.stft.wsin, layer.stft.wcos], "lr": 1e-4}]
    opt = torch.optim.SGD(groups)

    def logits(spec):                                            # (N, 256, W) or (N, 1, 64, 64): elementwise and sums only
        spec = spec.reshape(spec.shape[0], -1, spec.shape[-1]).mean(-1)
        return (spec * head[:spec.shape[1]]).sum(-1)
    grads_x = []
    for _ in range(steps):
        opt.zero_grad()
        if x.grad is not None:
            x.grad = None
        if case in ("radar", "stft"):
            loss = ((logits(layer(x)) - target) ** 2).mean() + ((logits(layer.forward_image(x, 64)) - target) ** 2).mean()
        else:
            loss = ((logits(layer.forward_upsampled(x, num_pad_frames=10, image_size=64)) - target) ** 2).mean()
        loss.backward()
        opt.step()
        if x.grad is not None:
            grads_x.append(x.grad.clone())
    params = [p.detach().clone() for grp in groups for p in grp["params"]]
    return params, grads_x


@pytest.mark.parametrize("case", ["radar", "stft", "ups_radar", "ups_stft"])
def test_module_sgd_steps_are_reproducible_under_deterministic_algorithms(case):
    before = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        p1, gx1 = _sgd_run(case)
        p2, gx2 = _sgd_run(case)
    finally:
        torch.use_deterministic_algorithms(before)
    assert len(p1) == len(p2)
    for a, b in zip(p1, p2):
        assert torch.isfinite(a).all()
        assert _same(a, b)
    for a, b in zip(gx1, gx2):
        assert _same(a, b)
    if case == "radar":
        assert len(gx1) == 3
