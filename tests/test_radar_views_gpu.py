"""Several radars per sequence (VirtualRadar.forward_views, C ABI VR_FLAG_VIEWS(R) with VR_FLAG_PER_SEQUENCE): R views of
each sequence of x (N, 3, T, V, M) in one launch equal, bit for bit, the per-sequence route on the repeated batch

    forward(x.repeat_interleave(R, 0), radar_location=loc.reshape(N*R, 3), wavelength=lam.reshape(N*R)).view(N, R, ...)

in every launch regime, and so do the placement gradients.  x is placed at the start of a NaN-filled allocation large enough
for N*R sequences: a kernel that read x through the output index instead of the x index would read NaN there and the
outputs would differ.  The unmarked tests at the end check the C ABI's argument handling without a GPU.

dL/dx for R > 1.  The kernel adds every view's float32 contributions to the entry's row in one running float32 sum, view by
view; the repeated route rounds each view's sum on its own and autograd adds the R results.  Per entry of joint v and body
m, a view adds k = 2 deg(v) float32 terms (one per bone end point in the bone loop, one in the mean-length loop; _counts).
The terms themselves are the same float32 values in both routes (same positions, placement and dL/d(iq) row).  With
u = 2^-24 and S = the sum of |term| over all R k terms (over-estimated by the oracle's per-path scale, which splits each
kernel term into its paths):
  * the views route, one recursive float32 sum of K = R k terms starting from an exact 0, is within (K - 1) u S of the exact
    sum of the terms;
  * view r of the repeated route is within (k - 1) u S_r of its exact sum, so the float64 sum of the R views (exact up to
    R 2^-53 S, negligible) is within (K - R) u S;
so |views - float64 sum of the repeated views| <= (2 K - R - 1) u S < 2 K u S.  The tests assert 2 K u S, plus 1e-12 S for
the float64 differences between the oracle's terms and the kernel's."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import backward as ob
from oracle import virtual_radar_oracle as vro
from tests.test_backward_property_gpu import U32, _counts, _scale
from tests.test_per_sequence_radar_gpu import FAR_L, LAMS, _batch, _edges, _same

RS = (1, 2, 3, 7)


def _cabi():
    from skeleton_action_recognition_b200 import _cabi
    return _cabi


def _layer(**kw):
    from skeleton_action_recognition_b200 import VirtualRadar
    return VirtualRadar(device="cuda", **kw).cuda()


@pytest.fixture
def schedule():
    cabi = _cabi()
    yield cabi.set_schedule
    cabi.set_schedule(-1)


def _views(N, R, seed=0, nan_view=None):
    """(wavelength (N, R), location (N, R, 3)): distinct per view, every third output (n R + r) exactly at the origin next
    to off-axis views of the same launch; nan_view = (n, r): that view far off-axis (the |u| > 1 bone of _batch)."""
    g = np.random.default_rng(seed)
    lam = np.array([[LAMS[(n + 3 * r) % len(LAMS)] for r in range(R)] for n in range(N)], np.float32)
    loc = (g.normal(size=(N, R, 3)) * 1.5).astype(np.float32)
    loc.reshape(-1, 3)[::3] = 0.0
    if nan_view is not None:
        loc[nan_view] = FAR_L
    return torch.from_numpy(lam), torch.from_numpy(loc)


def _guarded(x, R):
    """x on the GPU at the start of a NaN-filled allocation of N R sequences (standard-contiguous layout)."""
    N = x.shape[0]
    buf = torch.full((N * R,) + tuple(x.shape[1:]), float("nan"), device="cuda")
    buf[:N].copy_(x)
    return buf[:N]


def _guarded_fma(x, R):
    """The same for a coordinate-innermost x: the buffer is (N R, T, V, M, 3), x a permuted view of its first N rows."""
    N = x.shape[0]
    buf = torch.full((N * R,) + tuple(x.permute(0, 2, 3, 4, 1).shape[1:]), float("nan"), device="cuda")
    buf[:N].copy_(x.permute(0, 2, 3, 4, 1))
    return buf[:N].permute(0, 4, 1, 2, 3)


def _repeat(xg, R):
    """x.repeat_interleave(R, 0) in x's own layout (the layer picks the range rounding from the strides)."""
    if xg.stride(1) == 1:
        return xg.permute(0, 2, 3, 4, 1).repeat_interleave(R, 0).permute(0, 4, 1, 2, 3)
    return xg.repeat_interleave(R, 0)


def _repeated(run, layer, xg, lam, loc):
    N, R = loc.shape[:2]
    return run(layer, _repeat(xg, R), radar_location=loc.reshape(N * R, 3).cuda(), wavelength=lam.reshape(N * R).cuda())


def _views_equal_repeated(route, x, lam, loc, edges=vro.NTU_EDGES, layer_kw=None, ready=False, layout="planar"):
    """forward_views (route kwargs) on a NaN-guarded x vs. the per-sequence route on the repeated batch: bitwise."""
    N, R = loc.shape[:2]
    layer = _layer(edges=edges, **(layer_kw or {}))
    layer.assume_inputs_ready = ready
    xg = _guarded_fma(x.cuda(), R) if layout == "coordinate_innermost" else _guarded(x.cuda(), R)
    assert xg.data_ptr() == xg.untyped_storage().data_ptr()
    with torch.no_grad():
        out = layer.forward_views(xg, loc.cuda(), lam.cuda(), **route)
        if "num_pad_frames" in route:
            ref = layer.forward_upsampled(xg.repeat_interleave(R, 0), route["num_pad_frames"], route.get("sigma", 3),
                                          route.get("image_size"), radar_location=loc.reshape(N * R, 3).cuda(),
                                          wavelength=lam.reshape(N * R).cuda())
        elif "image_size" in route:
            ref = _repeated(lambda l, v, **kw: l.forward_image(v, route["image_size"], **kw), layer, xg, lam, loc)
        else:
            ref = _repeated(lambda l, v, **kw: l(v, **kw), layer, xg, lam, loc)
        if layout == "coordinate_innermost":      # forward() copies x to the planar layout: also check the launch itself
            xc = _guarded(xg.contiguous(), R)
            flags = _cabi().VR_FLAG_RANGE_FMA
            pl = layer._view_placements(xg, loc.cuda(), lam.cuda())
            assert _same(layer._run(xg, xc, flags, pl), ref)
    assert out.shape == (N, R) + tuple(ref.shape[-2:])
    assert _same(out.reshape(ref.shape), ref)
    return out


# ---- 1. forward: bitwise equal to the repeated per-sequence route ------------------------------------------------------------
CASES = {                     # (N, T, V, M, layout)
    "ntu": (5, 300, 25, 2, "planar"),
    "coordinate_innermost": (4, 300, 25, 2, "coordinate_innermost"),
    "one_body": (4, 300, 25, 1, "planar"),
    "three_bodies": (3, 300, 25, 3, "planar"),
    "generic_vm": (4, 256, 17, 2, "planar"),
    "long_park": (2, 5000, 25, 2, "planar"),
}


@pytest.mark.gpu
@pytest.mark.parametrize("R", RS)
@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("mode", [0, 1, "ready"])
def test_views_equal_the_repeated_batch(case, mode, R, schedule):
    N, T, V, M, layout = CASES[case]
    nan_seq = 1 if V == 25 else None
    x = _batch(N, T, V, M, seed=3, layout=layout, nan_seq=nan_seq)
    nan_view = (nan_seq, R - 1) if nan_seq is not None else None
    lam, loc = _views(N, R, seed=R, nan_view=nan_view)
    schedule(mode if mode != "ready" else -1)
    out = _views_equal_repeated({}, x, lam, loc, _edges(V), ready=mode == "ready", layout=layout)
    if nan_view is not None:      # the far view of the |u| > 1 sequence has NaN frames; every other view stays finite
        assert torch.isnan(out[nan_view]).any()
        for n in range(N):
            for r in range(R):
                if (n, r) != nan_view:
                    assert torch.isfinite(out[n, r]).all(), (n, r)


# More output jobs than CTAs / teams: every CTA and team runs several jobs from the ticket counter, and the views of one
# sequence land on different CTAs / teams.
BIG = {"ntu_many_jobs": (1300, 300), "park_many_jobs": (100, 5000)}


@pytest.mark.gpu
@pytest.mark.parametrize("R", RS)
@pytest.mark.parametrize("case", sorted(BIG))
@pytest.mark.parametrize("mode", [0, 1, "ready"])
def test_views_with_several_jobs_per_cta_and_team(case, mode, R, schedule):
    cabi = _cabi()
    NR, T = BIG[case]
    N = -(-NR // R)
    src, dst = map(list, zip(*vro.NTU_EDGES))
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    plan = cabi.plan(N * R, T, 25, 2, src, dst, sm_count=sms)
    assert N * R * plan["jobs_per_seq"] > 2 * plan["grid"]
    if case == "ntu_many_jobs":
        team = cabi.plan_team(N * R, T, 25, 2, src, dst, sm_count=sms)
        assert N * R > 2 * team["grid"] * team["teams_per_cta"]
    x = _batch(N, T, seed=16)
    lam, loc = _views(N, R, seed=11)
    schedule(mode if mode != "ready" else -1)
    out = _views_equal_repeated({}, x, lam, loc, ready=mode == "ready")
    assert torch.isfinite(out).all()


@pytest.mark.gpu
@pytest.mark.parametrize("R", RS)
@pytest.mark.parametrize("T", [300, 6000])            # F = 19 <= 256 columns, F = 376 > 256 (only kept frames)
def test_forward_image_views(T, R):
    x = _batch(3, T, seed=4)
    lam, loc = _views(3, R, seed=1)
    _views_equal_repeated(dict(image_size=256), x, lam, loc)


@pytest.mark.gpu
@pytest.mark.parametrize("R", RS)
@pytest.mark.parametrize("image_size", [None, 64])
@pytest.mark.parametrize("stft", ["fused", "general"])       # general: synthesis from the cubics, then the tcgen05 STFT
def test_forward_upsampled_views(image_size, R, stft):
    x = _batch(3, 24, seed=5)
    lam, loc = _views(3, R, seed=2)
    _views_equal_repeated(dict(num_pad_frames=40, sigma=3, image_size=image_size), x, lam, loc,
                          layer_kw=dict(train_stft_kernel=True) if stft == "general" else None)


@pytest.mark.gpu
@pytest.mark.parametrize("R", RS)
@pytest.mark.parametrize("n_fft", [128, 256, 512])
def test_general_stft_views(n_fft, R):
    x = _batch(3, 600, seed=6)
    lam, loc = _views(3, R, seed=3)
    _views_equal_repeated({}, x, lam, loc, layer_kw=dict(n_fft=n_fft, train_stft_kernel=True))
    _views_equal_repeated(dict(image_size=64), x, lam, loc, layer_kw=dict(n_fft=n_fft, train_stft_kernel=True))


@pytest.mark.gpu
def test_shared_placements_and_module_wavelength():
    """(R, 3) locations and (R,) / 0-d / absent wavelengths broadcast over the batch like their (N, R) expansions."""
    x = _batch(3, 300, seed=7).cuda()
    lam, loc = _views(1, 4, seed=4)
    layer = _layer(wavelength=9e-4)
    with torch.no_grad():
        full = layer.forward_views(x, loc[0].expand(3, 4, 3).cuda(), lam[0].expand(3, 4).cuda())
        assert torch.equal(layer.forward_views(x, loc[0].cuda(), lam[0].cuda()), full)
        ref = layer.forward_views(x, loc[0].expand(3, 4, 3).cuda(), torch.full((3, 4), 9e-4, device="cuda"))
        assert torch.equal(layer.forward_views(x, loc[0].cuda()), ref)
        assert torch.equal(layer.forward_views(x, loc[0].cuda(), torch.tensor(9e-4, device="cuda")), ref)
        assert layer.forward_views(x[:0], loc[0].cuda()).shape == (0, 4, 256, 19)


# ---- 2. gradients -----------------------------------------------------------------------------------------------------------------
def _route(route):
    if route.startswith("upsampled"):
        return dict(num_pad_frames=20, sigma=3)
    return {}


def _layer_kw(route):
    return dict(train_stft_kernel=True) if route in ("general", "upsampled_general") else {}


def _w(out):
    return torch.cos(torch.arange(out[0].numel(), device=out.device, dtype=torch.float32) * 0.37).view(out.shape[1:])


def _view_grads(route, x, lam, loc, stream=None):
    """forward_views + backward of sum(out * w) -> (dL/dlam (N, R), dL/dloc (N, R, 3), dL/dx or None, out)."""
    N, R = loc.shape[:2]
    layer = _layer(**_layer_kw(route))
    lam_t, loc_t = lam.cuda().requires_grad_(True), loc.cuda().requires_grad_(True)
    xg = x.cuda().requires_grad_(not route.startswith("upsampled"))
    if stream is not None:
        stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream if stream is not None else torch.cuda.current_stream()):
        out = layer.forward_views(xg, loc_t, lam_t, **_route(route))
        (out.reshape((N * R,) + out.shape[2:]) * _w(out.reshape((N * R,) + out.shape[2:]))).sum().backward()
    torch.cuda.synchronize()
    return lam_t.grad, loc_t.grad, xg.grad, out.detach()


def _repeated_grads(route, x, lam, loc):
    """The per-sequence route on the repeated batch -> (dL/dlam (N R,), dL/dloc (N R, 3), per-view dL/dx (N R, ...), out)."""
    N, R = loc.shape[:2]
    layer = _layer(**_layer_kw(route))
    lam_t = lam.reshape(N * R).cuda().requires_grad_(True)
    loc_t = loc.reshape(N * R, 3).cuda().requires_grad_(True)
    xr = x.cuda().repeat_interleave(R, 0).requires_grad_(not route.startswith("upsampled"))
    if route.startswith("upsampled"):
        out = layer.forward_upsampled(xr, 20, 3, radar_location=loc_t, wavelength=lam_t)
    else:
        out = layer(xr, radar_location=loc_t, wavelength=lam_t)
    (out * _w(out)).sum().backward()
    torch.cuda.synchronize()
    return lam_t.grad, loc_t.grad, xr.grad, out.detach()


@pytest.mark.gpu
@pytest.mark.parametrize("R", RS)
@pytest.mark.parametrize("route", ["fused", "general", "upsampled", "upsampled_general"])
def test_view_gradients_equal_the_repeated_batch(route, R):
    """Placement gradients: the repeated route's bits (a per-output gradient does not depend on its batch position).  dL/dx:
    bitwise with R = 1; for R > 1, deterministic and close to the sum of the repeated route's per-view gradients (the
    bound is tested against the oracle's term magnitudes in test_view_synthesis_adjoint_against_the_oracle)."""
    N = 3
    T = 24 if route.startswith("upsampled") else 300
    x = _batch(N, T, seed=8)
    lam, loc = _views(N, R, seed=4 + R)
    gl, gL, gx, out = _view_grads(route, x, lam, loc)
    rl, rL, rx, rout = _repeated_grads(route, x, lam, loc)
    assert torch.equal(out.reshape(rout.shape), rout)
    assert torch.equal(gl.reshape(N * R), rl) and torch.equal(gL.reshape(N * R, 3), rL)
    assert torch.isfinite(gl).all() and (gl != 0).all()
    if gx is None:
        return
    if R == 1:
        assert torch.equal(gx, rx)
    else:
        ref = rx.double().view((N, R) + tuple(x.shape[1:])).sum(1)
        scale = rx.double().abs().view((N, R) + tuple(x.shape[1:])).sum(1)
        # A sanity bound only.  The per-entry bound 2 K 2^-24 sum|terms| of the module docstring needs the terms' magnitudes,
        # which only the oracle provides; test_view_synthesis_adjoint_against_the_oracle asserts it through
        # vr_synth_adjoint_f32.  It covers this path: the fused and general backward compute dL/dx in the same kernel
        # (vr_synth_adjoint_ps_kernel<false, true>) from a dL/d(iq) that is the repeated route's bits row by row (the
        # adjoint STFT and the general STFT backward are per output), so only the views' float32 accumulation differs.
        assert ((gx.double() - ref).abs() <= 1e-4 * scale.amax() + 1e-3 * scale).all()
    # repeated call and another stream: the same bits
    for other in (_view_grads(route, x, lam, loc), _view_grads(route, x, lam, loc, stream=torch.cuda.Stream())):
        assert torch.equal(other[0], gl) and torch.equal(other[1], gL) and torch.equal(other[2], gx)
    # a sequence's gradients do not depend on the rest of the batch
    perm = torch.tensor([2, 0, 1])
    pl, pL, px, _ = _view_grads(route, x[perm], lam[perm], loc[perm])
    assert torch.equal(pl, gl[perm.cuda()]) and torch.equal(pL, gL[perm.cuda()]) and torch.equal(px, gx[perm.cuda()])
    sl, sL, sx, _ = _view_grads(route, x[1:2], lam[1:2], loc[1:2])
    assert torch.equal(sl, gl[1:2]) and torch.equal(sL, gL[1:2]) and torch.equal(sx, gx[1:2])


def _synth_adjoint_views(x, giq, lam, loc, flags, R):
    """vr_synth_adjoint_f32 with VR_FLAG_PER_SEQUENCE | VR_FLAG_VIEWS(R) on a NaN-guarded x -> (gradients (N R, 4) float64,
    dL/dx (N, ...))."""
    cabi = _cabi()
    xg = _guarded(x.cuda(), R)
    gg = giq.cuda().contiguous()
    lam_d, loc_d = lam.reshape(-1).cuda(), loc.reshape(-1, 3).cuda()
    N, _, T, V, M = xg.shape
    gp = torch.zeros(cabi.per_sequence_grad_doubles(N * R, T), dtype=torch.float64, device="cuda")
    gx = torch.empty_like(xg)
    src, dst = map(list, zip(*vro.NTU_EDGES))
    cabi.check(cabi.lib().vr_synth_adjoint_f32(xg.data_ptr(), gg.data_ptr(), N * R, T, V, M, cabi.i32_array(src),
                                               cabi.i32_array(dst), len(src), lam_d.data_ptr(), loc_d.data_ptr(),
                                               flags | cabi.VR_FLAG_PER_SEQUENCE | cabi.views_flag(R), gp.data_ptr(),
                                               gx.data_ptr(), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    return gp[:4 * N * R].view(N * R, 4), gx


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["seq", "fma"])
@pytest.mark.parametrize("R", [2, 3])
def test_view_synthesis_adjoint_against_the_oracle(mode, R):
    """vr_synth_adjoint_f32 with views: each output's parameter gradients are the bits of the plain per-sequence call on the
    repeated batch and within oracle/backward.py's tolerances; dL/dx is within the module docstring's bound of the float64
    sum of the repeated call's per-view dL/dx, and within R times the stage tolerance of the oracle summed over the views."""
    from tests.test_backward_property_gpu import compare, tolerances
    from tests.test_per_sequence_radar_gpu import _synth_adjoint_ps
    N, T = 2, 200
    x = _batch(N, T, seed=10)
    giq = torch.randn(N * R, T, 2, generator=torch.Generator().manual_seed(11))
    lam, loc = _views(N, R, seed=6)
    flags = _cabi().VR_FLAG_RANGE_FMA if mode == "fma" else 0
    g, gx = _synth_adjoint_views(x, giq, lam, loc, flags, R)
    rg, rx = _synth_adjoint_ps(x.repeat_interleave(R, 0), giq, lam.reshape(-1), loc.reshape(-1, 3), flags)
    assert torch.equal(g, rg)
    k = _counts(vro.NTU_EDGES, 25)[:, None]              # float32 additions per view into an entry of joint v
    for n in range(N):
        refs = [ob.synth_adjoint(x[n:n + 1].numpy(), giq[n * R + r:n * R + r + 1].numpy(), vro.NTU_EDGES,
                                 float(lam[n, r]), tuple(loc[n, r].tolist()), mode) for r in range(R)]
        for r, ref in enumerate(refs):
            got = (float(g[n * R + r, 0]), g[n * R + r, 1:].cpu().numpy(), rx[n * R + r:n * R + r + 1].cpu().numpy().astype(np.float64))
            compare("%s/R%d/%d.%d" % (mode, R, n, r), got, ref, tolerances(ref, vro.NTU_EDGES))
        S = sum(_scale(ref, "x") for ref in refs)
        got_x = gx[n:n + 1].cpu().numpy().astype(np.float64)
        rep = rx[n * R:(n + 1) * R].cpu().numpy().astype(np.float64).sum(0, keepdims=True)
        bound = 2 * R * k * U32 * S + 1e-12 * S
        assert (np.abs(got_x - rep) <= bound).all(), float((np.abs(got_x - rep) / np.maximum(bound, 1e-300)).max())
        oracle_x = sum(ref["x"] for ref in refs)
        assert (np.abs(got_x - oracle_x) <= 4 * R * k * U32 * S + 1e-12 * S).all()
    # deterministic
    g2, gx2 = _synth_adjoint_views(x, giq, lam, loc, flags, R)
    assert torch.equal(g2, g) and torch.equal(gx2, gx)


@pytest.mark.gpu
def test_view_gradients_replay_in_a_cuda_graph():
    cabi = _cabi()
    N, R, T = 3, 3, 300
    x = _guarded(_batch(N, T, seed=12).cuda(), R)
    lam, loc = [t.cuda() for t in _views(N, R, seed=7)]
    lam, loc = lam.reshape(-1), loc.reshape(-1, 3)
    layer = _layer()
    flags = cabi.VR_FLAG_PER_SEQUENCE | cabi.views_flag(R)
    out, iq = layer._launch(x, flags, want_iq=True, lam=lam, loc=loc)
    assert out.shape[0] == N * R
    go = torch.randn(out.shape, generator=torch.Generator().manual_seed(3)).cuda()
    gz = torch.empty_like(iq)
    gp = torch.zeros(cabi.per_sequence_grad_doubles(N * R, T), dtype=torch.float64, device="cuda")
    gx = torch.empty_like(x)
    src, dst = map(list, zip(*vro.NTU_EDGES))
    sc, dc = cabi.i32_array(src), cabi.i32_array(dst)

    def step():
        gp.zero_()
        cabi.check(cabi.lib().vr_backward_f32(x.data_ptr(), iq.data_ptr(), go.data_ptr(), N * R, T, 25, 2, sc, dc, len(src),
                                              lam.data_ptr(), loc.data_ptr(), 256, 16, flags, gz.data_ptr(), gp.data_ptr(),
                                              gx.data_ptr(), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    step()
    torch.cuda.synchronize()
    eager, eager_x = gp[:4 * N * R].clone(), gx.clone()
    assert torch.isfinite(eager_x).all()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    for _ in range(3):
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(gp[:4 * N * R], eager) and torch.equal(gx, eager_x)


@pytest.mark.gpu
def test_views_of_raw_sequences_need_a_detached_x():
    layer = _layer()
    x = _batch(2, 24).cuda().requires_grad_(True)
    with pytest.raises(NotImplementedError):
        layer.forward_views(x, torch.zeros(2, 3, device="cuda"), num_pad_frames=10)
    with torch.no_grad():
        assert layer.forward_views(x, torch.zeros(2, 3, device="cuda"), num_pad_frames=10).shape == (2, 2, 256, 16)


# ---- 3. errors ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_bad_view_placements_raise():
    layer = _layer()
    x = _batch(4, 300).cuda()
    loc = torch.zeros(4, 3, 3, device="cuda")
    with pytest.raises(ValueError):
        layer.forward_views(x, loc, torch.full((2,), 1e-3, device="cuda"))          # R = 3 locations, 2 wavelengths
    with pytest.raises(ValueError):
        layer.forward_views(x, loc, torch.full((4, 2), 1e-3, device="cuda"))
    with pytest.raises(ValueError):
        layer.forward_views(x, torch.zeros(3, device="cuda"))                       # 1-D
    with pytest.raises(ValueError):
        layer.forward_views(x, torch.zeros(5, 3, 3, device="cuda"))                 # wrong N
    with pytest.raises(ValueError):
        layer.forward_views(x, torch.zeros(4, 0, 3, device="cuda"))                 # R = 0
    with pytest.raises(ValueError):
        layer.forward_views(x, torch.zeros(256, 3, device="cuda"))                  # R > 255
    with pytest.raises(ValueError):
        layer.forward_views(x, torch.zeros(4, 3, 2, device="cuda"))                 # (N, R, 2)
    with pytest.raises(ValueError):
        layer.forward_views(x, loc.double())                                          # float64
    with pytest.raises(ValueError):
        layer.forward_views(x, loc, torch.full((3,), 1e-3, device="cuda", dtype=torch.float64))
    with pytest.raises(RuntimeError):
        layer.forward_views(x, loc.cpu())                                             # CPU tensor
    with pytest.raises(RuntimeError):
        layer.forward_views(x, loc, torch.full((3,), 1e-3))
    if torch.cuda.device_count() > 1:                                                 # another device
        with pytest.raises(RuntimeError):
            layer.forward_views(x, loc.to("cuda:1"))
    with pytest.raises(ValueError):
        layer.forward_views(x, loc, image_size=0)


class _ViewsModule(torch.nn.Module):
    def __init__(self, layer):
        super().__init__()
        self.layer = layer

    def forward(self, x, loc, lam):
        return self.layer.forward_views(x, loc, lam)


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two CUDA devices")
def test_data_parallel_scatters_the_view_placements():
    layer = _layer()
    x = _batch(6, 300, seed=15).cuda()
    lam, loc = [t.cuda() for t in _views(6, 3, seed=10)]
    with torch.no_grad():
        one = layer.forward_views(x, loc, lam)
        dp = torch.nn.DataParallel(_ViewsModule(layer), device_ids=[0, 1])(x, loc, lam)
    assert torch.equal(dp, one)


# ---- C ABI without a GPU ----------------------------------------------------------------------------------------------------------
def test_cabi_rejects_bad_views():
    cabi = _cabi()
    L = cabi.lib()
    src, dst = map(list, zip(*vro.NTU_EDGES))
    sc, dc = cabi.i32_array(src), cabi.i32_array(dst)
    ps = cabi.VR_FLAG_PER_SEQUENCE
    fake = ctypes.c_void_p(256)                     # never dereferenced: the checks come first
    args = lambda N, flags: (fake, N, 300, 25, 2, sc, dc, len(src), fake, fake, 256, 16, flags, fake, None)   # noqa: E731
    # views without per-sequence placements
    assert L.vr_forward_f32(*args(6, cabi.views_flag(3))) == cabi.VR_ERR_ARG
    assert "VR_FLAG_PER_SEQUENCE" in cabi.last_error()
    assert L.vr_backward_f32(fake, fake, fake, 6, 300, 25, 2, sc, dc, len(src), fake, fake, 256, 16, cabi.views_flag(3), fake,
                             fake, None, None) == cabi.VR_ERR_ARG
    # N not a multiple of R
    assert L.vr_forward_f32(*args(7, ps | cabi.views_flag(3))) == cabi.VR_ERR_SHAPE
    assert L.vr_forward_image_f32(fake, 7, 300, 25, 2, sc, dc, len(src), fake, fake, 256, 16, ps | cabi.views_flag(2), 64,
                                  fake, None) == cabi.VR_ERR_SHAPE
    assert L.vr_synth_f32(fake, 5, 300, 25, 2, sc, dc, len(src), fake, fake, ps | cabi.views_flag(2), fake, None) == cabi.VR_ERR_SHAPE
    assert L.vr_synth_adjoint_f32(fake, fake, 5, 300, 25, 2, sc, dc, len(src), fake, fake, ps | cabi.views_flag(2), fake, None,
                                  None) == cabi.VR_ERR_SHAPE
    assert L.vr_backward_params_f32(fake, fake, fake, 9, 300, 25, 2, sc, dc, len(src), fake, fake, 256, 16,
                                    ps | cabi.views_flag(2), fake, fake, None) == cabi.VR_ERR_SHAPE
    assert L.vr_synth_adjoint_upsampled_f32(fake, fake, 5, 24, 25, 2, sc, dc, len(src), fake, fake, ps | cabi.views_flag(2),
                                            10, fake, None) == cabi.VR_ERR_SHAPE
    assert L.vr_backward_upsampled_params_f32(fake, fake, fake, 5, 24, 25, 2, sc, dc, len(src), fake, fake, 256, 16,
                                              ps | cabi.views_flag(2), 10, fake, fake, None) == cabi.VR_ERR_SHAPE
    # the field beyond 8 bits is an unknown flag
    assert L.vr_forward_f32(*args(6, ps | (256 << cabi.VR_FLAG_VIEWS_SHIFT))) == cabi.VR_ERR_ARG
    # R = 0 has no flag value
    with pytest.raises(ValueError):
        cabi.views_flag(0)
    with pytest.raises(ValueError):
        cabi.views_flag(256)
    assert cabi.views_of(ps) == 1 and cabi.views_of(ps | cabi.views_flag(7)) == 7
    # the host entry takes one placement for the batch
    x = np.zeros((1, 3, 300, 25, 2), np.float32)
    out = np.zeros((1, 256, 19), np.float32)
    loc = (ctypes.c_float * 3)(0, 0, 0)
    for flags in (cabi.views_flag(1), ps | cabi.views_flag(1)):
        assert L.vr_forward_host_f32(x.ctypes.data, 1, 300, 25, 2, sc, dc, len(src), ctypes.c_float(1e-3), loc, 256, 16, flags,
                                     out.ctypes.data, 0) == cabi.VR_ERR_ARG
        assert "VR_FLAG_VIEWS" in cabi.last_error()


def test_cabi_sizes_the_upsampling_workspace_by_raw_sequences():
    """The _upsampled entries solve the spline once per raw sequence: a workspace for N / R sequences is enough, one byte
    less is rejected before anything reaches the device."""
    cabi = _cabi()
    L = cabi.lib()
    src, dst = map(list, zip(*vro.NTU_EDGES))
    sc, dc = cabi.i32_array(src), cabi.i32_array(dst)
    fake = ctypes.c_void_p(256)
    flags = cabi.VR_FLAG_PER_SEQUENCE | cabi.views_flag(3)
    need = int(L.vr_upsampled_workspace_bytes(2, 24, 25, 2))
    assert need * 3 == int(L.vr_upsampled_workspace_bytes(6, 24, 25, 2))
    for fn in (lambda nb: L.vr_forward_upsampled_f32(fake, 6, 24, 25, 2, sc, dc, len(src), fake, fake, 256, 16, flags, 10,
                                                     ctypes.c_float(3.0), 0, fake, nb, fake, None),
               lambda nb: L.vr_synth_upsampled_f32(fake, 6, 24, 25, 2, sc, dc, len(src), fake, fake, flags, 10,
                                                   ctypes.c_float(3.0), fake, nb, fake, None)):
        assert fn(need - 1) == cabi.VR_ERR_ARG
        assert "vr_upsampled_workspace_bytes = %d" % need in cabi.last_error()
