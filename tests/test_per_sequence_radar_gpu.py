"""Per-sequence radar placements (VR_FLAG_PER_SEQUENCE; the `radar_location=` / `wavelength=` keywords of
VirtualRadar.forward, forward_image and forward_upsampled): one launch that sees sequence n from radar_location[n] at
wavelength[n] equals, bit for bit, a layer with those scalar parameters run on x[n:n+1] -- in both schedules, under
VR_FLAG_INPUTS_READY, in every kernel variant -- and its per-sequence gradients are the same bits wherever the sequence
sits in the batch.  The unmarked tests at the end check the C ABI's argument handling without a GPU."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import backward as ob
from oracle import virtual_radar_oracle as vro

LAMS = (5e-4, 9e-4, 1e-3, 5e-3)
FAR_L = (30.0, -20.0, 40.0)         # far off-axis: bones of 1 m pointing at it round to |u| > 1 a third of the time
U_BONE = (0, 1)                     # NTU bone 0 -> 1 (the first spine bone) is made to point at FAR_L


def _cabi():
    from skeleton_action_recognition_b200 import _cabi
    return _cabi


def _layer(**kw):
    from skeleton_action_recognition_b200 import VirtualRadar
    return VirtualRadar(device="cuda", **kw).cuda()


@pytest.fixture
def schedule():
    """Sets the forward schedule for one test and restores the default (automatic) afterwards."""
    cabi = _cabi()
    yield cabi.set_schedule
    cabi.set_schedule(-1)


# ---- inputs ---------------------------------------------------------------------------------------------------------------
def _fma32(a, b, c):
    return np.float32(np.float64(a) * np.float64(b) + np.float64(c))


def _norm2(v, fma):
    """Squared norm as the forward rounds it: "seq" ((x x + y y) + z z) or, for coordinate-innermost inputs, FMA."""
    if fma:
        return _fma32(v[2], v[2], _fma32(v[1], v[1], v[0] * v[0]))
    return (v[0] * v[0] + v[1] * v[1]) + v[2] * v[2]


def _u2_f32(S, D, L, fma=False):
    """The forward's squared aspect cosine of the bone S -> D in float32, op by op."""
    f = np.float32
    S, D, L = [np.asarray(v, np.float32) for v in (S, D, L)]
    B, A = D - S, f(2) * L - (S + D)
    bb, aa = _norm2(B, fma), _norm2(A, fma)
    ab = (A[0] * B[0] + A[1] * B[1]) + A[2] * B[2]
    u = ab / (np.sqrt(aa) * np.sqrt(bb) + f(2e-6))
    return u * u


def _u_gt_one_bone(seed=0):
    """(S, D): a 1 m bone pointing at FAR_L whose float32 aspect cosine rounds to |u| > 1 (acos -> NaN in the reference)."""
    rng = np.random.default_rng(seed)
    L = np.asarray(FAR_L, np.float32)
    for _ in range(1000):
        S = (rng.normal(size=3) * 0.3).astype(np.float32)
        d = (L - S) / np.linalg.norm(L - S)
        D = (S + d.astype(np.float32)).astype(np.float32)
        if _u2_f32(S, D, L) > 1 and _u2_f32(S, D, L, fma=True) > 1:      # NaN in both range modes
            return S, D
    raise AssertionError("no |u| > 1 bone found")


def _placements(N, seed=0, nan_seq=None):
    """Distinct (wavelength, location) per sequence: wavelengths from LAMS, every third location exactly at the origin
    (the kernels' fast path), the others off-axis, sequence 1 far off-axis."""
    g = np.random.default_rng(seed)
    lam = np.array([LAMS[n % len(LAMS)] for n in range(N)], np.float32)
    loc = (g.normal(size=(N, 3)) * 1.5).astype(np.float32)
    loc[::3] = 0.0
    if N > 1:
        loc[1] = (6.0, -3.0, 7.0)
    if nan_seq is not None:
        loc[nan_seq] = FAR_L
    return torch.from_numpy(lam), torch.from_numpy(loc)


def _batch(N, T=300, V=25, M=2, seed=0, layout="planar", nan_seq=None):
    g = torch.Generator().manual_seed(seed)
    if layout == "coordinate_innermost":
        x = (torch.randn(N, T, V, M, 3, generator=g) * 0.3).permute(0, 4, 1, 2, 3)
    else:
        x = torch.randn(N, 3, T, V, M, generator=g) * 0.3
    if nan_seq is not None:
        S, D = _u_gt_one_bone()
        x = x.clone() if layout == "planar" else x.contiguous()
        x[nan_seq, :, T // 2, U_BONE[0], 0] = torch.from_numpy(S)
        x[nan_seq, :, T // 2, U_BONE[1], 0] = torch.from_numpy(D)
        if layout == "coordinate_innermost":
            x = x.permute(0, 2, 3, 4, 1).contiguous().permute(0, 4, 1, 2, 3)
    return x


def _edges(V):
    if V == 25:
        return vro.NTU_EDGES
    return [(i, (i * 7 + 3) % V if (i * 7 + 3) % V != i else (i + 1) % V) for i in range(V)]


def _per_sequence_equals_single(run, x, lam, loc, edges, **layer_kw):
    """run(layer, x, radar_location=, wavelength=) on the batch vs. one scalar layer per sequence on x[n:n+1]: bitwise."""
    layer = _layer(edges=edges, **layer_kw)
    xg = x.cuda()
    with torch.no_grad():
        out = run(layer, xg, radar_location=loc.cuda(), wavelength=lam.cuda())
        for n in range(x.shape[0]):
            one = _layer(edges=edges, wavelength=float(lam[n]), radar_location=loc[n].tolist(), **layer_kw)
            ref = run(one, xg[n:n + 1])
            assert _same(out[n:n + 1], ref), n
    return out


def _same(a, b):
    """Bitwise equal, NaN where the other is NaN (a NaN compares unequal to itself)."""
    na, nb = torch.isnan(a), torch.isnan(b)
    return torch.equal(na, nb) and torch.equal(torch.where(na, 0.0, a), torch.where(nb, 0.0, b))


# ---- 1. bitwise equal to one layer per sequence -----------------------------------------------------------------------------
CASES = {                     # (N, T, V, M, layout)
    "ntu": (8, 300, 25, 2, "planar"),
    "coordinate_innermost": (6, 300, 25, 2, "coordinate_innermost"),
    "one_body": (6, 300, 25, 1, "planar"),
    "three_bodies": (5, 300, 25, 3, "planar"),
    "generic_vm": (6, 256, 17, 2, "planar"),
    "long_park": (4, 5000, 25, 2, "planar"),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("mode", [0, 1, "ready"])
def test_forward_equals_one_layer_per_sequence(case, mode, schedule):
    N, T, V, M, layout = CASES[case]
    nan_seq = 2 if V == 25 else None
    x = _batch(N, T, V, M, seed=3, layout=layout, nan_seq=nan_seq)
    lam, loc = _placements(N, nan_seq=nan_seq)
    schedule(mode if mode != "ready" else -1)

    def run(layer, xg, **kw):
        layer.assume_inputs_ready = mode == "ready"
        return layer(xg, **kw)

    out = _per_sequence_equals_single(run, x, lam, loc, _edges(V))
    if nan_seq is not None:      # the |u| > 1 sequence has NaN frames; its neighbours stay finite
        assert torch.isnan(out[nan_seq]).any()
        for n in range(N):
            if n != nan_seq:
                assert torch.isfinite(out[n]).all(), n


# Batches with more jobs than CTAs / teams: every CTA (cooperative schedule) or team (team-job schedule) runs several jobs,
# drawn from the launch's ticket counter, and switches from one sequence's placement to another's.  Sequences that land on
# later jobs -- the tail of the batch, and a stride through it -- are checked against the scalar single-sequence layer.
BIG = {"ntu_many_jobs": (1300, 300), "park_many_jobs": (100, 5000)}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(BIG))
@pytest.mark.parametrize("mode", [0, 1, "ready"])
def test_forward_with_several_jobs_per_cta_and_team(case, mode, schedule):
    cabi = _cabi()
    N, T = BIG[case]
    src, dst = map(list, zip(*vro.NTU_EDGES))
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    plan = cabi.plan(N, T, 25, 2, src, dst, sm_count=sms)
    assert N * plan["jobs_per_seq"] > 2 * plan["grid"]          # every CTA of the cooperative schedule loops
    if case == "ntu_many_jobs":
        team = cabi.plan_team(N, T, 25, 2, src, dst, sm_count=sms)
        assert N > 2 * team["grid"] * team["teams_per_cta"]       # every team runs at least two jobs
    x = _batch(N, T, seed=16)
    lam, loc = _placements(N, seed=11)
    schedule(mode if mode != "ready" else -1)
    layer = _layer()
    layer.assume_inputs_ready = mode == "ready"
    xg = x.cuda()
    with torch.no_grad():
        out = layer(xg, radar_location=loc.cuda(), wavelength=lam.cuda())
        sample = sorted(set([0, 1, 2] + list(range(N - 6, N)) + list(range(7, N, max(N // 16, 1))) + list(range(N // 2, N, 41))))
        for n in sample:
            one = _layer(wavelength=float(lam[n]), radar_location=loc[n].tolist())
            assert _same(out[n:n + 1], one(xg[n:n + 1])), n
    assert torch.isfinite(out).all()


@pytest.mark.gpu
def test_per_sequence_gradients_of_a_large_batch():
    """More (sequence, segment) units than warps in the grid, so that the warps of the reduction loop: the gradients of a
    few sequences are the bits they have in a batch of four."""
    N = 2000
    x = _batch(N, 300, seed=17)
    lam, loc = _placements(N, seed=12)
    gl, gL, gx = _layer_grads("fused", x, lam, loc)
    idx = torch.tensor([0, 1, 1500, N - 1])
    sl, sL, sx = _layer_grads("fused", x[idx], lam[idx], loc[idx])
    assert torch.equal(sl, gl[idx.cuda()]) and torch.equal(sL, gL[idx.cuda()]) and torch.equal(sx, gx[idx.cuda()])


@pytest.mark.gpu
@pytest.mark.parametrize("T", [300, 6000])            # F = 19 <= 256 columns, F = 376 > 256 (only kept frames)
def test_forward_image_equals_one_layer_per_sequence(T):
    x = _batch(4, T, seed=4)
    lam, loc = _placements(4, seed=1)
    _per_sequence_equals_single(lambda layer, xg, **kw: layer.forward_image(xg, 256, **kw), x, lam, loc, vro.NTU_EDGES)


@pytest.mark.gpu
@pytest.mark.parametrize("image_size", [None, 64])
def test_forward_upsampled_equals_one_layer_per_sequence(image_size):
    x = _batch(4, 24, seed=5)
    lam, loc = _placements(4, seed=2)
    _per_sequence_equals_single(lambda layer, xg, **kw: layer.forward_upsampled(xg, 40, 3, image_size, **kw),
                                x, lam, loc, vro.NTU_EDGES)


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft", [128, 256, 512])
def test_general_stft_equals_one_layer_per_sequence(n_fft):
    x = _batch(4, 600, seed=6)
    lam, loc = _placements(4, seed=3)
    _per_sequence_equals_single(lambda layer, xg, **kw: layer(xg, **kw), x, lam, loc, vro.NTU_EDGES,
                                n_fft=n_fft, train_stft_kernel=True)


# ---- 2. broadcast identity ----------------------------------------------------------------------------------------------------
def _route_kw(route):
    return dict(train_stft_kernel=True) if route == "general" else {}


def _route_run(route, layer, xg, **kw):
    if route == "upsampled":
        return layer.forward_upsampled(xg, 20, 3, **kw)
    return layer(xg, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("route", ["fused", "general", "upsampled"])
def test_expanded_module_parameters_equal_the_scalar_call(route):
    T = 24 if route == "upsampled" else 300
    x = _batch(4, T, seed=7).cuda()
    grads = []
    for per_seq in (False, True):
        layer = _layer(wavelength=9e-4, radar_location=[0.4, -0.7, 1.3], train_wavelength=True, train_radar_location=True,
                       **_route_kw(route))
        xg = x.clone().requires_grad_(route != "upsampled")
        kw = {}
        if per_seq:
            kw = dict(radar_location=layer.radar_location.expand(4, 3), wavelength=layer.wavelength.expand(4))
            for t in kw.values():
                t.retain_grad()
        out = _route_run(route, layer, xg, **kw)
        out.square().mean().backward()
        grads.append((out.detach(), xg.grad, layer.wavelength.grad, layer.radar_location.grad))
    (o0, gx0, gl0, gL0), (o1, gx1, gl1, gL1) = grads
    assert torch.equal(o0, o1)
    if route != "upsampled":
        assert torch.equal(gx0, gx1)
    # the module-parameter gradients are now autograd's float32 sum of the per-sequence gradients: equal up to the
    # rounding of that sum (a few units in the last place of the sum of magnitudes)
    per_lam, per_loc = kw["wavelength"].grad, kw["radar_location"].grad
    assert per_lam.shape == (4,) and per_loc.shape == (4, 3)
    assert float((gl1 - gl0).abs()) <= 1e-6 * float(per_lam.abs().sum())
    assert ((gL1 - gL0).abs() <= 1e-6 * per_loc.abs().sum(0)).all()


# ---- 3. gradients ---------------------------------------------------------------------------------------------------------------
def _layer_grads(route, x, lam, loc, stream=None):
    """forward + backward of loss = sum(out * w) with per-sequence placements -> (dL/dlam (N,), dL/dloc (N,3), dL/dx)."""
    layer = _layer(**_route_kw(route))
    lam_t = lam.cuda().requires_grad_(True)
    loc_t = loc.cuda().requires_grad_(True)
    xg = x.cuda().requires_grad_(route != "upsampled")
    if stream is not None:
        stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream if stream is not None else torch.cuda.current_stream()):
        out = _route_run(route, layer, xg, radar_location=loc_t, wavelength=lam_t)
        w = torch.cos(torch.arange(out[0].numel(), device=out.device, dtype=torch.float32) * 0.37).view(out.shape[1:])
        (out * w).sum().backward()
    torch.cuda.synchronize()
    return lam_t.grad, loc_t.grad, xg.grad


@pytest.mark.gpu
@pytest.mark.parametrize("route", ["fused", "general", "upsampled"])
def test_per_sequence_gradients_do_not_depend_on_the_batch(route):
    N = 6
    T = 24 if route == "upsampled" else 300
    x = _batch(N, T, seed=8)
    lam, loc = _placements(N, seed=4)
    gl, gL, gx = _layer_grads(route, x, lam, loc)
    assert torch.isfinite(gl).all() and torch.isfinite(gL).all() and (gl != 0).all()
    # repeated call, another stream
    again = _layer_grads(route, x, lam, loc)
    side = _layer_grads(route, x, lam, loc, stream=torch.cuda.Stream())
    for other in (again, side):
        assert torch.equal(other[0], gl) and torch.equal(other[1], gL)
        if gx is not None:
            assert torch.equal(other[2], gx)
    # the same sequences at other batch positions, and in a smaller batch
    perm = torch.tensor([3, 0, 5, 1, 4, 2])
    pl, pL, px = _layer_grads(route, x[perm], lam[perm], loc[perm])
    assert torch.equal(pl, gl[perm.cuda()]) and torch.equal(pL, gL[perm.cuda()])
    sl, sL, sx = _layer_grads(route, x[2:4], lam[2:4], loc[2:4])
    assert torch.equal(sl, gl[2:4]) and torch.equal(sL, gL[2:4])
    if gx is not None:
        assert torch.equal(px, gx[perm.cuda()]) and torch.equal(sx, gx[2:4])
        # dL/dx: bitwise the single-sequence scalar call's
        for n in range(N):
            layer = _layer(wavelength=float(lam[n]), radar_location=loc[n].tolist(), **_route_kw(route))
            xn = x[n:n + 1].cuda().requires_grad_(True)
            out = layer(xn)
            w = torch.cos(torch.arange(out[0].numel(), device=out.device, dtype=torch.float32) * 0.37).view(out.shape[1:])
            (out * w).sum().backward()
            assert torch.equal(xn.grad, gx[n:n + 1]), n


@pytest.mark.gpu
@pytest.mark.parametrize("route", ["fused", "general", "upsampled"])
def test_per_sequence_gradients_match_the_scalar_path(route):
    """Against the scalar path on each sequence alone (a different float64 summation order, the same float32 result up to
    its last place); the float64 values themselves are checked against the oracle below."""
    N = 4
    T = 24 if route == "upsampled" else 300
    x = _batch(N, T, seed=9)
    lam, loc = _placements(N, seed=5)
    gl, gL, _ = _layer_grads(route, x, lam, loc)
    for n in range(N):
        layer = _layer(wavelength=float(lam[n]), radar_location=loc[n].tolist(), train_wavelength=True,
                       train_radar_location=True, **_route_kw(route))
        out = _route_run(route, layer, x[n:n + 1].cuda())
        w = torch.cos(torch.arange(out[0].numel(), device=out.device, dtype=torch.float32) * 0.37).view(out.shape[1:])
        (out * w).sum().backward()
        # both are float64 totals rounded to float32: at most one unit in the last place apart
        torch.testing.assert_close(gl[n], layer.wavelength.grad, rtol=2 ** -22, atol=0)
        torch.testing.assert_close(gL[n], layer.radar_location.grad, rtol=2 ** -22, atol=1e-9 * float(gL[n].abs().max()))


def _synth_adjoint_ps(x, giq, lam, loc, flags):
    cabi = _cabi()
    xg, gg = x.cuda().contiguous(), giq.cuda().contiguous()
    lam_d, loc_d = lam.cuda(), loc.cuda()           # held until the launch has read them
    N, _, T, V, M = xg.shape
    gp = torch.zeros(cabi.per_sequence_grad_doubles(N, T), dtype=torch.float64, device="cuda")
    gx = torch.empty_like(xg)
    src, dst = map(list, zip(*vro.NTU_EDGES))
    cabi.check(cabi.lib().vr_synth_adjoint_f32(xg.data_ptr(), gg.data_ptr(), N, T, V, M, cabi.i32_array(src),
                                               cabi.i32_array(dst), len(src), lam_d.data_ptr(), loc_d.data_ptr(),
                                               flags | cabi.VR_FLAG_PER_SEQUENCE, gp.data_ptr(), gx.data_ptr(),
                                               ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    return gp[:4 * N].view(N, 4), gx


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["seq", "fma"])
def test_per_sequence_synthesis_adjoint_against_the_oracle(mode):
    """vr_synth_adjoint_f32 with the flag, sequence by sequence against oracle/backward.py's synth_adjoint and against the
    scalar call on that sequence alone, with the stage-level tolerances of tests/test_backward_property_gpu.py."""
    from tests.test_backward_property_gpu import compare, synth_gpu, tolerances
    N, T = 3, 200
    x = _batch(N, T, seed=10)
    giq = torch.randn(N, T, 2, generator=torch.Generator().manual_seed(11))
    lam, loc = _placements(N, seed=6)
    flags = _cabi().VR_FLAG_RANGE_FMA if mode == "fma" else 0
    g, gx = _synth_adjoint_ps(x, giq, lam, loc, flags)
    for n in range(N):
        ref = ob.synth_adjoint(x[n:n + 1].numpy(), giq[n:n + 1].numpy(), vro.NTU_EDGES, float(lam[n]),
                               tuple(loc[n].tolist()), mode)
        got = (float(g[n, 0]), g[n, 1:].cpu().numpy(), gx[n:n + 1].cpu().numpy().astype(np.float64))
        tols = tolerances(ref, vro.NTU_EDGES)
        compare("%s/%d" % (mode, n), got, ref, tols)
        gp1, gx1 = synth_gpu(x[n:n + 1], giq[n:n + 1], vro.NTU_EDGES, float(lam[n]), tuple(loc[n].tolist()), flags)
        assert torch.equal(gx1, gx[n:n + 1].cuda())          # dL/dx: bitwise the scalar call's
        assert abs(float(gp1[0]) - got[0]) <= 2 * tols[0], n
        assert (np.abs(gp1[1:].cpu().numpy() - got[1]) <= 2 * tols[1]).all(), n


@pytest.mark.gpu
def test_per_sequence_gradients_replay_in_a_cuda_graph():
    cabi = _cabi()
    N, T = 4, 300
    x = _batch(N, T, seed=12).cuda()
    lam, loc = [t.cuda() for t in _placements(N, seed=7)]
    layer = _layer()
    flags = cabi.VR_FLAG_PER_SEQUENCE
    out, iq = layer._launch(x, flags, want_iq=True, lam=lam, loc=loc)
    go = torch.randn(out.shape, generator=torch.Generator().manual_seed(3)).cuda()
    gz = torch.empty_like(iq)
    gp = torch.zeros(cabi.per_sequence_grad_doubles(N, T), dtype=torch.float64, device="cuda")
    src, dst = map(list, zip(*vro.NTU_EDGES))
    sc, dc = cabi.i32_array(src), cabi.i32_array(dst)

    def step():
        gp.zero_()
        cabi.check(cabi.lib().vr_backward_params_f32(x.data_ptr(), iq.data_ptr(), go.data_ptr(), N, T, 25, 2, sc, dc, len(src),
                                                     lam.data_ptr(), loc.data_ptr(), 256, 16, flags, gz.data_ptr(),
                                                     gp.data_ptr(), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    step()
    torch.cuda.synchronize()
    eager = gp[:4 * N].clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()                                  # warm-up on the capture stream
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    for _ in range(3):
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(gp[:4 * N], eager)


@pytest.mark.gpu
def test_deterministic_algorithms_need_nothing_more():
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        x = _batch(3, 300, seed=13)
        lam, loc = _placements(3, seed=8)
        a = _layer_grads("fused", x, lam, loc)
        b = _layer_grads("fused", x, lam, loc)
    finally:
        torch.use_deterministic_algorithms(prev)
    assert all(torch.equal(p, q) for p, q in zip(a, b))


# ---- 4. errors -------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_bad_placements_raise():
    layer = _layer()
    x = _batch(4, 300).cuda()
    ok_loc, ok_lam = torch.zeros(4, 3, device="cuda"), torch.full((4,), 1e-3, device="cuda")
    with pytest.raises(ValueError):
        layer(x, radar_location=torch.zeros(5, 3, device="cuda"))            # wrong N
    with pytest.raises(ValueError):
        layer(x, wavelength=torch.full((3,), 1e-3, device="cuda"))
    with pytest.raises(ValueError):
        layer(x, radar_location=torch.zeros(4, 2, device="cuda"))            # (N, 2)
    with pytest.raises(ValueError):
        layer(x, radar_location=ok_loc.double())                             # float64
    with pytest.raises(ValueError):
        layer.forward_image(x, 64, wavelength=ok_lam.double())
    with pytest.raises(RuntimeError):
        layer(x, radar_location=ok_loc.cpu())                                # CPU tensor
    with pytest.raises(RuntimeError):
        layer.forward_upsampled(x[:, :, :20], 10, 3, wavelength=ok_lam.cpu())
    if torch.cuda.device_count() > 1:                                        # another device
        with pytest.raises(RuntimeError):
            layer(x, radar_location=ok_loc.to("cuda:1"))
    with pytest.raises(TypeError):
        layer.forward_host(x.cpu(), radar_location=ok_loc)
    with pytest.raises(TypeError):
        layer.forward_notebook(torch.zeros(20, 25, 3, device="cuda"), wavelength=ok_lam)


@pytest.mark.gpu
def test_model_passes_placements_through():
    from skeleton_action_recognition_b200.models.resnet import Model
    model = Model(num_classes=5, num_filters=8, image_size=64, device="cuda").cuda().eval()
    x = _batch(3, 300, seed=14).cuda()
    lam, loc = [t.cuda() for t in _placements(3, seed=9)]
    with torch.no_grad():
        img = model.spectrogram_image(x, radar_location=loc, wavelength=lam)
        ref = model.virtual_radar.forward_image(x, 64, radar_location=loc, wavelength=lam)
        assert torch.equal(img, ref)
        assert model(x, radar_location=loc, wavelength=lam).shape == (3, 5)


# ---- 5. multi-GPU -----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two CUDA devices")
def test_data_parallel_scatters_the_placements():
    layer = _layer()
    x = _batch(6, 300, seed=15).cuda()
    lam, loc = [t.cuda() for t in _placements(6, seed=10)]
    with torch.no_grad():
        one = layer(x, radar_location=loc, wavelength=lam)
        dp = torch.nn.DataParallel(layer, device_ids=[0, 1])(x, radar_location=loc, wavelength=lam)
    assert torch.equal(dp, one)


# ---- C ABI without a GPU ----------------------------------------------------------------------------------------------------------
def test_cabi_rejects_the_flag_without_device_arrays():
    cabi = _cabi()
    L = cabi.lib()
    src, dst = map(list, zip(*vro.NTU_EDGES))
    sc, dc = cabi.i32_array(src), cabi.i32_array(dst)
    flag = cabi.VR_FLAG_PER_SEQUENCE
    fake = ctypes.c_void_p(256)                     # never dereferenced: the checks come first
    # null placement pointers: rejected by the entries' own null checks, with or without the flag (pins that behaviour)
    assert L.vr_forward_f32(fake, 2, 300, 25, 2, sc, dc, len(src), None, None, 256, 16, flag, fake, None) == cabi.VR_ERR_ARG
    assert L.vr_synth_f32(fake, 2, 300, 25, 2, sc, dc, len(src), None, fake, flag, fake, None) == cabi.VR_ERR_ARG
    assert L.vr_backward_f32(fake, fake, fake, 2, 300, 25, 2, sc, dc, len(src), None, None, 256, 16, flag, fake, fake,
                             None, None) == cabi.VR_ERR_ARG
    # a per-sequence gradient buffer that is not 8-byte aligned
    assert L.vr_backward_f32(fake, fake, fake, 2, 300, 25, 2, sc, dc, len(src), fake, fake, 256, 16, flag, fake,
                             ctypes.c_void_p(260), None, None) == cabi.VR_ERR_ARG
    assert "aligned" in cabi.last_error()
    # the host-buffer entry takes one placement for the batch
    x = np.zeros((1, 3, 300, 25, 2), np.float32)
    out = np.zeros((1, 256, 19), np.float32)
    loc = (ctypes.c_float * 3)(0, 0, 0)
    assert L.vr_forward_host_f32(x.ctypes.data, 1, 300, 25, 2, sc, dc, len(src), ctypes.c_float(1e-3), loc, 256, 16, flag,
                                 out.ctypes.data, 0) == cabi.VR_ERR_ARG
    assert "VR_FLAG_PER_SEQUENCE" in cabi.last_error()


@pytest.mark.parametrize("N,T", [(1, 1), (3, 32), (3, 33), (256, 300), (16, 75000)])
def test_per_sequence_grad_buffer_size(N, T):
    cabi = _cabi()
    n = cabi.per_sequence_grad_doubles(N, T)
    segs = -(-T // 32)
    assert n == 4 * N + 4 * N * segs                # N x 4 gradients, then 4 partials per (sequence, 32-step segment)
    assert cabi.per_sequence_grad_doubles(0, T) == 0 and cabi.per_sequence_grad_doubles(N, 0) == 0
