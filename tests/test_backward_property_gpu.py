"""The backward pass (csrc/vr_backward.cuh) against a float32-phase adjoint oracle, over arbitrary skeletons, layouts, hops
and lengths.

dL/dx and dL/d(radar_location) are the sum of three paths: the phase (through the range d), the aspect cosine u and the
mean bone length.  The two amplitude paths are 1e-4 .. 1e-2 of the phase path, so a comparison with float32 autograd
(tests/test_backward_gpu.py) cannot see them.  `oracle.backward.synth_adjoint` makes the kernel's deliberate roundings --
float32 range, phase and mean bone length, float64 for the rest -- so the kernel and the oracle differ only by float64
round-off and by the float32 stores of dL/dx.  The tolerances follow from that:

  parameters   1e-12 * (sum of |term| over every (sequence, step, bone, body) term of the gradient);
  dL/dx        per entry 4 * k * 2^-24 * (sum over the bones touching it of |contribution|), k = the number of float32
               additions the kernel makes into that entry (two per bone end point).

The CPU tests below pin the oracle (to the float64 closed form and to float64 autograd at the float32 operating point)
and show, on the fixed cases the GPU tests run, that these tolerances are at least 10x below every path and reject
deliberately wrong variants of the oracle.  The GPU tests print, per case, the achieved error over the tolerance and the
smallest path over the tolerance."""
import ctypes

import numpy as np
import pytest
import torch
from hypothesis import HealthCheck, given, settings, strategies as st

from oracle import backward as ob
from oracle import virtual_radar_oracle as vro
from tests import fixtures as fx

U32 = 2.0 ** -24
FAR = [(0., 0., 5.), (6., -3., 7.), (2., 9., -4.)]          # the body offsets of test_far_targets_large_phase
OFF_AXIS = (0.5, -1.0, 2.0)


# ---- inputs -----------------------------------------------------------------------------------------------------------
def _edges(kind, V, E, pick):
    """The four kinds of bone list of tests/test_property_gpu.py; `pick(lo, hi)` draws an integer."""
    if kind == "star":
        hub = pick(0, V - 1)
        edges = [(hub, (hub + 1 + i) % V) for i in range(E)]
    elif kind == "chain":
        edges = [(i % V, (i + 1) % V) for i in range(E)]
    elif kind == "duplicates":
        a, b = pick(0, V - 1), pick(0, V - 1)
        b = b if b != a else (a + 1) % V
        edges = ([(a, b), (a, b), (b, a)] + [(pick(0, V - 1), pick(0, V - 1)) for _ in range(max(E - 3, 0))])[:E]
    else:
        edges = [(pick(0, V - 1), pick(0, V - 1)) for _ in range(E)]
    return [(s, d if d != s else (s + 1) % V) for s, d in edges]       # a zero-length bone is 0/0 in the reference


@st.composite
def skeletons(draw, max_E=40, big_E=False, star_cap=None):
    V = draw(st.integers(2, 34))
    M = draw(st.integers(1, 4))
    E = 128 if big_E and draw(st.integers(0, 7)) == 0 else draw(st.integers(1, max_E))
    kind = draw(st.sampled_from(["random", "star", "chain", "duplicates"]))
    if kind == "star" and star_cap:      # the forward puts every bone of a star into one bone group
        E = min(E, star_cap)
    return V, M, _edges(kind, V, E, lambda lo, hi: draw(st.integers(lo, hi)))


def _positions(shape, seed, offset=None, layout="planar", scale=0.4):
    """(N,3,T,V,M) float32 joint positions; "coordinate_innermost" is a permuted view of an (N,T,V,M,3) tensor."""
    N, _, T, V, M = shape
    g = torch.Generator().manual_seed(seed)
    if layout == "coordinate_innermost":
        x = (torch.randn(N, T, V, M, 3, generator=g) * scale).permute(0, 4, 1, 2, 3)
    else:
        x = torch.randn(N, 3, T, V, M, generator=g) * scale
    if offset is not None:
        x = x + torch.tensor(offset, dtype=torch.float32).view(1, 3, 1, 1, 1)
        if layout == "coordinate_innermost":
            x = x.permute(0, 2, 3, 4, 1).contiguous().permute(0, 4, 1, 2, 3)
    return x


def _counts(edges, V):
    """float32 additions into each dL/dx entry of joint v: one per bone end point in the bone loop, one in the mean-length
    loop."""
    src, dst = map(list, zip(*edges))
    return 2 * np.bincount(np.array(src + dst), minlength=V)


def _scale(ref, k):
    return sum(ref["scale"][p][k] for p in ob.PATHS)


def tolerances(ref, edges):
    """The stage-level tolerances of the module docstring: (lam, loc (3,), x (N,3,T,V,M))."""
    V = ref["x"].shape[3]
    k = _counts(edges, V)[:, None]
    sx = _scale(ref, "x")
    return 1e-12 * _scale(ref, "lam"), 1e-12 * _scale(ref, "loc"), 4 * k * U32 * sx + 1e-12 * sx


def _ratio(diff, tol):
    """max |diff| / tol; an entry with tol == 0 must have diff == 0 exactly (inf otherwise)."""
    diff, tol = np.abs(np.asarray(diff, np.float64)), np.broadcast_to(tol, np.shape(diff))
    if np.any((tol == 0) & (diff != 0)):
        return np.inf
    sel = tol > 0
    return float((diff[sel] / tol[sel]).max()) if sel.any() else 0.0


def _path_margins(ref, tols):
    """Smallest max |path| / tol over the paths that carry a gradient: how far above the tolerance each path sits."""
    out = {}
    for p in ob.PATHS:
        for k, t in zip(("lam", "loc", "x"), tols):
            if np.abs(ref["paths"][p][k]).max() > 0:
                out["%s/%s" % (p, k)] = _ratio(ref["paths"][p][k], t)
    return out


def compare(tag, got, ref, tols):
    """got = (lam, loc, x) of the kernel; asserts every error <= its tolerance and prints the margins."""
    errs = [_ratio(g - r, t) for g, r, t in zip(got, (ref["lam"], ref["loc"], ref["x"]), tols)]
    margins = _path_margins(ref, tols)
    smallest = min(margins, key=margins.get) if margins else None
    print("%s: error/tolerance lam %.2e loc %.2e x %.2e | smallest path/tolerance %s %.2e"
          % (tag, errs[0], errs[1], errs[2], smallest, margins.get(smallest, np.nan)))
    assert errs[0] <= 1 and errs[1] <= 1 and errs[2] <= 1, (tag, errs)
    return errs, margins


# ---- the GPU entry points ------------------------------------------------------------------------------------------------
def _lib():
    from skeleton_action_recognition_b200 import _cabi
    return _cabi


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _params(lam, loc):
    return (torch.tensor(float(np.float32(lam)), dtype=torch.float32, device="cuda"),
            torch.tensor(np.float32(loc), dtype=torch.float32, device="cuda"))


def synth_gpu(x, giq, edges, lam, loc, flags, want_x=True):
    """vr_synth_adjoint_f32 -> (gparams float64 (4,), dL/dx float32 or None), both on the GPU."""
    cabi = _lib()
    xg = x if x.is_cuda else x.cuda()
    xg = xg.contiguous()
    gg = giq.cuda().contiguous() if not giq.is_cuda else giq.contiguous()
    N, _, T, V, M = xg.shape
    lam_t, loc_t = _params(lam, loc)
    gp = torch.zeros(4, dtype=torch.float64, device="cuda")
    gx = torch.empty_like(xg) if want_x else None
    src, dst = map(list, zip(*edges))
    cabi.check(cabi.lib().vr_synth_adjoint_f32(xg.data_ptr(), gg.data_ptr(), N, T, V, M, cabi.i32_array(src),
                                               cabi.i32_array(dst), len(src), lam_t.data_ptr(), loc_t.data_ptr(), flags,
                                               gp.data_ptr(), gx.data_ptr() if want_x else None, _stream()))
    return gp, gx


def backward_gpu(x, iq, go, edges, lam, loc, hop, flags, want_x=True):
    """vr_backward_f32 -> (dL/d(iq) float32, gparams float64, dL/dx or None), on the GPU."""
    cabi = _lib()
    N, _, T, V, M = x.shape
    lam_t, loc_t = _params(lam, loc)
    gz = torch.empty(N, T, 2, dtype=torch.float32, device="cuda")
    gp = torch.zeros(4, dtype=torch.float64, device="cuda")
    gx = torch.empty_like(x) if want_x else None
    src, dst = map(list, zip(*edges))
    cabi.check(cabi.lib().vr_backward_f32(x.data_ptr(), iq.data_ptr(), go.data_ptr(), N, T, V, M, cabi.i32_array(src),
                                          cabi.i32_array(dst), len(src), lam_t.data_ptr(), loc_t.data_ptr(), 256, hop, flags,
                                          gz.data_ptr(), gp.data_ptr(), gx.data_ptr() if want_x else None, _stream()))
    return gz, gp, gx


def stft_adjoint_tolerance(iq, go, hop, n_fft=256):
    """Per-sample bound on the float32 error of the adjoint STFT (vr_stft_adjoint_kernel), from the conditioning of each
    frame: the radix FFT of the windowed frame zp errs by at most eps_X = 2 u log2(n) sum |zp| per bin, and
    G = g X / |X|^2 turns that into |g| eps_X / |X|^2 (large where a bin nearly vanishes); the inverse FFT adds
    2 u log2(n) sum |G|, the window and the float32 overlap-add, in the owner form's fixed frame order,
    u * (frames + 2) * sum |y|.  A coarse bound for these end-to-end cases; tests/test_backward_oracle_gpu.py holds the
    kernel to a bound derived from its instructions.  Stage 2 propagates the error actually measured."""
    iq = np.asarray(iq, np.float64)
    g = np.asarray(go, np.float64)
    N, T, _ = iq.shape
    z = iq[..., 0] + 1j * iq[..., 1]
    n = np.arange(n_fft)
    w = 0.5 - 0.5 * np.cos(2 * np.pi * n / n_fft)
    c = 2 * U32 * np.log2(n_fft)
    bound, mag = np.zeros((N, T)), np.zeros((N, T))
    F = T // hop + 1
    for f in range(F):
        idx = ob._reflect(f * hop - n_fft // 2 + n, T)
        zp = z[:, idx] * w
        X = np.fft.fft(zp, axis=1)
        a = np.abs(X)
        gk = np.roll(g[:, :, f], -(n_fft // 2), axis=1)
        with np.errstate(divide="ignore", invalid="ignore"):
            sens = np.where(a > 0, np.abs(gk) / (a * a), 0)
            G = np.where(a > 0, gk * X / (a * (a + 1e-6) + (a == 0)), 0)
        eps_X = c * np.abs(zp).sum(1, keepdims=True)
        per = (sens * eps_X).sum(1, keepdims=True) + c * np.abs(G).sum(1, keepdims=True)
        y = np.abs(w * (np.fft.ifft(G, axis=1) * n_fft))
        np.add.at(bound, (slice(None), idx), w * per)
        np.add.at(mag, (slice(None), idx), y)
    frames = -(-n_fft // hop)
    return (bound + U32 * (frames + 2) * mag)[..., None]


def check_stft_adjoint(tag, gz, iq, go, hop):
    """dL/d(iq) of the GPU against ob.stft_adjoint within stft_adjoint_tolerance -> (float64 dL/d(iq), |error|)."""
    iq, go = iq.cpu().numpy(), go.cpu().numpy()
    want = ob.stft_adjoint(iq, go, hop=hop)
    err = np.abs(gz.cpu().numpy().astype(np.float64) - want)
    r = _ratio(err, stft_adjoint_tolerance(iq, go, hop))
    print("%s: dL/d(iq) error %.2e of its max, %.2e of its tolerance" % (tag, err.max() / np.abs(want).max(), r))
    assert r <= 1, (tag, r)
    return want, err


def _flags(mode):
    return _lib().VR_FLAG_RANGE_FMA if mode == "fma" else 0


def check_stage(tag, x, giq, edges, lam, loc, mode, repeat=False):
    """vr_synth_adjoint_f32 against synth_adjoint on (x, giq) with the stage-level tolerances."""
    xc = x.contiguous()
    gp, gx = synth_gpu(xc, giq, edges, lam, loc, _flags(mode))
    ref = ob.synth_adjoint(xc.numpy(), giq.numpy(), edges, lam, loc, mode)
    got = (float(gp[0]), gp[1:].cpu().numpy(), gx.cpu().numpy().astype(np.float64))
    compare(tag, got, ref, tolerances(ref, edges))
    if repeat:
        _, gx2 = synth_gpu(xc, giq, edges, lam, loc, _flags(mode))
        assert torch.equal(gx, gx2), "dL/dx differs between two identical launches"
    return ref, got


# ---- fixed cases: run on the GPU (test_fixed_cases_stage_level), and their sensitivity proven on the CPU --------------------
def _ntu_case(kw, seed):
    """The inputs of test_gradient_wrt_the_skeleton_data: s3_smooth, T = 200; dL/d(iq) of the float64 closed form."""
    x = fx.s3_smooth(2, T=200)
    go = torch.randn(2, 256, 13, generator=torch.Generator().manual_seed(seed)).numpy()
    _, _, iq = ob.analytic_grads(x.numpy(), go, **kw)
    return x, torch.from_numpy(ob.stft_adjoint(iq, go).astype(np.float32)), vro.NTU_EDGES


def _random_case(shape, edges, seed, layout="planar", offset=None):
    x = _positions(shape, seed, offset, layout)
    giq = torch.randn(shape[0], shape[2], 2, generator=torch.Generator().manual_seed(seed + 1))
    return x, giq, edges


def _fixed(name):
    """name -> (x, giq, edges, wavelength, radar_location)."""
    if name == "ntu_lam5e-3_origin":
        return _ntu_case(dict(wavelength=5e-3), 7) + (5e-3, (0., 0., 0.))
    if name == "ntu_lam1e-3_offaxis":
        return _ntu_case(dict(wavelength=1e-3, radar_location=(0.3, -0.2, 1.5)), 7) + (1e-3, (0.3, -0.2, 1.5))
    if name == "star_M3_coordinate_innermost":
        return _random_case((2, 3, 300, 9, 3), [(4, v) for v in range(9) if v != 4] + [(0, 1), (1, 2)], 31,
                            "coordinate_innermost") + (9e-4, OFF_AXIS)
    if name == "chain_far":
        return _random_case((2, 3, 257, 12, 1), [(i, i + 1) for i in range(11)], 32, offset=FAR[1]) + (5e-4, (0., 0., 0.))
    raise KeyError(name)


FIXED = ["ntu_lam5e-3_origin", "ntu_lam1e-3_offaxis", "star_M3_coordinate_innermost", "chain_far"]


# ---- CPU: the oracle pinned ------------------------------------------------------------------------------------------------
@settings(max_examples=25, deadline=None, derandomize=True, suppress_health_check=[HealthCheck.too_slow, HealthCheck.data_too_large])
@given(sk=skeletons(max_E=30), N=st.integers(1, 2), T=st.sampled_from([129, 160, 250]), hop=st.sampled_from([8, 16, 37]),
       loc=st.sampled_from([(0., 0., 0.), (0.3, -0.2, 1.5)]), lam=st.sampled_from([5e-4, 5e-3]), seed=st.integers(0, 2 ** 16))
def test_oracle_in_float64_equals_the_closed_form(sk, N, T, hop, loc, lam, seed):
    """With theta and the mean bone length in float64, synth_adjoint(x, stft_adjoint(iq, go)) is analytic_grads."""
    V, M, edges = sk
    x = _positions((N, 3, T, V, M), seed).numpy()
    go = torch.randn(N, 256, T // hop + 1, generator=torch.Generator().manual_seed(seed)).numpy()
    kw = dict(edges=edges, wavelength=lam, radar_location=loc, hop_length=hop)
    g_lam, g_loc, iq = ob.analytic_grads(x, go, **kw)
    _, _, g_x = ob.analytic_grads(x, go, wrt_x=True, **kw)
    ref = ob.synth_adjoint(x, ob.stft_adjoint(iq, go, hop=hop), edges, lam, loc, theta32=False, cbar32=False)
    assert _ratio(ref["lam"] - g_lam, 1e-12 * _scale(ref, "lam")) <= 1
    assert _ratio(ref["loc"] - g_loc, 1e-12 * _scale(ref, "loc")) <= 1
    assert _ratio(ref["x"] - g_x, 1e-12 * _scale(ref, "x")) <= 1


def autograd_at_float32_phase(x, giq, edges, lam, loc, mode, substitute=True):
    """float64 torch autograd of the reference's graph (layers/virtual_radar.py:93-123) in which the phase and the mean bone
    length take the float32 values of the forward: theta = theta64 + (theta32 - theta64).detach(), likewise cbar (the mean
    then weighs the lengths with f32(1/E), as the kernel does).  substitute=False: the plain float64 graph."""
    src, dst = map(list, zip(*edges))
    x64 = torch.from_numpy(np.asarray(x, np.float64)).requires_grad_(True)
    lam64 = torch.tensor(float(np.float32(lam)), dtype=torch.float64, requires_grad=True)
    loc64 = torch.tensor(np.float32(loc).astype(np.float64), requires_grad=True)
    S, D, L = x64[:, :, :, src], x64[:, :, :, dst], loc64[:, None, None, None]
    th64 = 4 * np.pi * torch.norm(torch.abs(S - L), dim=1) / lam64
    _, th32 = vro.range_phase_c(torch.from_numpy(np.asarray(x, np.float32)[:, :, :, src]), np.float32(loc), np.float32(lam), mode)
    th = th64 + (th32.double() - th64).detach() if substitute else th64
    A, B = L - (S + D) / 2, D - S
    cosang = torch.sum(A * B, dim=1) / (torch.norm(A, dim=1) * torch.norm(B, dim=1) + 1e-6)
    aspect = torch.acos(cosang)
    azim = torch.asin((loc64[1] - S[:, 1]) / (torch.norm(torch.abs(S - L)[:, :2], dim=1) + 1e-6))
    cbar64 = torch.norm(S - D, dim=1).sum(2, keepdim=True) * (float(np.float32(1) / np.float32(len(src))) if substitute
                                                               else 1.0 / len(src))
    ln = ob._bone_lengths_f32(np.asarray(x, np.float32)[:, :, :, src], np.asarray(x, np.float32)[:, :, :, dst], mode)
    sumB = np.zeros(ln.shape[:2] + ln.shape[3:], np.float32)
    for e in range(len(src)):
        sumB = sumB + ln[:, :, e]
    cbar32 = torch.from_numpy((sumB * (np.float32(1) / np.float32(len(src)))).astype(np.float64))[:, :, None]
    cbar = cbar64 + (cbar32 - cbar64).detach() if substitute else cbar64
    semi = cbar ** 2
    sin2 = torch.sin(aspect) ** 2
    denom = sin2 * torch.cos(azim) ** 2 + sin2 * torch.sin(azim) ** 2 + semi * torch.cos(aspect) ** 2
    amp = torch.sqrt(np.pi * semi / denom ** 2)
    iq = torch.stack(((amp * torch.cos(th)).sum((2, 3)), (amp * torch.sin(th)).sum((2, 3))), -1)
    loss = (iq * torch.from_numpy(np.asarray(giq, np.float64))).sum()
    g = torch.autograd.grad(loss, (lam64, loc64, x64))
    return float(g[0]), g[1].numpy(), g[2].numpy()


@pytest.mark.parametrize("layout", ["planar", "coordinate_innermost"])
@pytest.mark.parametrize("case", [
    dict(V=25, M=2, edges=vro.NTU_EDGES, lam=5e-3, loc=(0., 0., 0.), offset=None),
    dict(V=7, M=3, edges=[(2, v) for v in range(7) if v != 2] + [(0, 1), (0, 1)], lam=1e-3, loc=(0.3, -0.2, 1.5), offset=None),
    dict(V=10, M=1, edges=[(i, i + 1) for i in range(9)], lam=5e-4, loc=(0., 0., 0.), offset=FAR[0]),
])
def test_oracle_equals_float64_autograd_at_the_float32_phase(case, layout):
    """An independent check of every derivative, by torch autograd of the reference's ops.
      * theta and cbar in float64 (theta32=False, cbar32=False): the oracle is the plain float64 graph's gradient to 1e-12
        of sum |term|, on every path -- the amplitude paths included, whose margin over this tolerance is printed.
      * at the kernel's operating point (float32 theta and cbar substituted with .detach()): the oracle's derivative factors
        differ from the graph's only where the kernel takes a float32 value -- d in 4 pi / (lambda d), theta in
        -theta / lambda, f32(1/E) -- by at most a few 2^-24 of each term of the phase and mean-length paths.  Those paths
        get 2^-21 of their sum |term|, everything else 1e-12.
    (With theta in float64, the two graphs round theta = 1e3 .. 1e5 rad differently: 4 theta 2^-53 more.)"""
    N, T = 2, 180
    x = _positions((N, 3, T, case["V"], case["M"]), 41, case["offset"], layout).contiguous().numpy()
    mode = "fma" if layout == "coordinate_innermost" else "seq"
    giq = torch.randn(N, T, 2, generator=torch.Generator().manual_seed(42)).numpy()
    args = (x, giq, case["edges"], case["lam"], case["loc"], mode)
    theta_max = 4 * np.pi * np.linalg.norm(x - np.float32(case["loc"])[:, None, None, None], axis=1).max() / case["lam"]
    for sub in (False, True):
        ref = ob.synth_adjoint(*args, theta32=sub, cbar32=sub)
        auto = autograd_at_float32_phase(*args, substitute=sub)
        sc = ref["scale"]
        for k, a in zip(("lam", "loc", "x"), auto):
            # float64 theta: one rounding of theta (1e3 .. 1e5 rad) moves cos and sin by theta * 2^-53
            loose = 2.0 ** -21 * (sc["phase"][k] + sc["length"][k]) if sub else 4 * theta_max * 2.0 ** -53 * _scale(ref, k)
            tol = loose + 1e-12 * _scale(ref, k)
            r = _ratio(ref[k] - a, tol)
            amp = {p: _ratio(ref["paths"][p][k], tol) for p in ("u", "length") if np.abs(ref["paths"][p][k]).max() > 0}
            print("%s %s %s: |oracle - autograd| / tolerance %.2e; amplitude paths / tolerance %s"
                  % (layout, "float32 theta" if sub else "float64", k, r, {p: "%.1e" % v for p, v in amp.items()}))
            assert r <= 1, (sub, k, r)
            if not sub:
                assert all(v >= 10 for v in amp.values()), (k, amp)


@pytest.mark.parametrize("name", FIXED)
def test_tolerances_see_every_path_and_reject_wrong_oracles(name):
    """The written proof that the GPU tests can fail: on each fixed case the stage-level tolerance is at least 10x below the
    largest contribution of each path, and each deliberately wrong oracle -- mean-length path removed, u path removed,
    theta in float64, the other range mode -- misses the right one by at least 10x the tolerance."""
    x, giq, edges, lam, loc = _fixed(name)
    mode = vro.distance_mode_for(x)
    xc = x.contiguous().numpy()
    ref = ob.synth_adjoint(xc, giq.numpy(), edges, lam, loc, mode)
    tols = tolerances(ref, edges)
    margins = _path_margins(ref, tols)
    print(name, {k: "%.1e" % v for k, v in margins.items()})
    assert set(margins) >= {"phase/lam", "phase/loc", "phase/x", "u/loc", "u/x", "length/x"}, margins
    assert min(margins.values()) >= 10, margins
    other = "seq" if mode == "fma" else "fma"
    variants = {
        "no mean-length path": {k: ref[k] - ref["paths"]["length"][k] for k in ("lam", "loc", "x")},
        "no u path": {k: ref[k] - ref["paths"]["u"][k] for k in ("lam", "loc", "x")},
        "theta in float64": ob.synth_adjoint(xc, giq.numpy(), edges, lam, loc, mode, theta32=False),
        "range mode %s" % other: ob.synth_adjoint(xc, giq.numpy(), edges, lam, loc, other),
    }
    for vname, v in variants.items():
        miss = max(_ratio(v[k] - ref[k], t) for k, t in zip(("lam", "loc", "x"), tols))
        print("  %s: rejected at %.1e x the tolerance" % (vname, miss))
        assert miss >= 10, (name, vname, miss)


# ---- GPU: stage level ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", FIXED)
def test_fixed_cases_stage_level(name):
    x, giq, edges, lam, loc = _fixed(name)
    check_stage(name, x, giq, edges, lam, loc, vro.distance_mode_for(x), repeat=True)


@pytest.mark.gpu
@settings(max_examples=30, deadline=None, derandomize=True, suppress_health_check=[HealthCheck.too_slow, HealthCheck.data_too_large])
@given(sk=skeletons(big_E=True), N=st.integers(1, 5), T=st.sampled_from([1, 2, 7, 64, 129, 300, 777, 1500]),
       lam=st.sampled_from([5e-4, 9e-4, 1e-3, 5e-3]), where=st.sampled_from(["origin", "off-axis", "far"]),
       fma=st.booleans(), seed=st.integers(0, 2 ** 16))
def test_synthesis_adjoint_property(sk, N, T, lam, where, fma, seed):
    """vr_synth_adjoint_f32 on arbitrary skeletons (V 2-34, M 1-4, E 1-40 and 128, four kinds of bone list), T 1-1500 (this
    entry has no T minimum), radar at the origin, off-axis or 5-10 m away (theta > 1e5 rad), both range modes."""
    V, M, edges = sk
    if N * T * len(edges) * M > 3_000_000:                    # keeps the CPU oracle within a second or two
        N = 1
    offset = FAR[seed % 3] if where == "far" else None
    loc = OFF_AXIS if where == "off-axis" else (0., 0., 0.)
    x = _positions((N, 3, T, V, M), seed, offset)
    giq = torch.randn(N, T, 2, generator=torch.Generator().manual_seed(seed + 7))
    tag = "V=%d M=%d E=%d N=%d T=%d lam=%g %s %s" % (V, M, len(edges), N, T, lam, where, "fma" if fma else "seq")
    check_stage(tag, x, giq, edges, lam, loc, "fma" if fma else "seq", repeat=True)


# ---- GPU: the module end to end ------------------------------------------------------------------------------------------------
def _layer(edges, lam, loc, hop, **kw):
    from skeleton_action_recognition_b200 import VirtualRadar
    return VirtualRadar(edges=edges, wavelength=lam, radar_location=list(loc), hop_length=hop, device="cuda:0", **kw).to("cuda:0")


def check_module(tag, x, edges, lam, loc, hop, seed):
    """The module's backward (x.requires_grad, both parameters trainable) in two stages:
      1. dL/d(iq) of vr_backward_f32 on the GPU's own saved iq against ob.stft_adjoint (stft_adjoint_tolerance);
      2. the module's gradients against synth_adjoint(x, float64 dL/d(iq)).  The tolerance adds to the stage-level one the
         propagated error of dL/d(iq) (float32 FFT and atomics): twice the measured per-sequence max error delta, pushed
         through the oracle as sum |term| with dL/d(iq) = (delta, 0) and (0, delta).  The module returns its parameter
         gradients in float32, which adds 2^-24 of their value."""
    cabi = _lib()
    mode = vro.distance_mode_for(x)
    layer = _layer(edges, lam, loc, hop, train_wavelength=True, train_radar_location=True)
    xg = x.cuda().requires_grad_(True)
    assert vro.distance_mode_for(xg) == mode
    out = layer(xg)
    go = torch.randn(out.shape, generator=torch.Generator().manual_seed(seed)).cuda()
    (out * go).sum().backward()
    assert xg.grad.stride() == xg.stride()                  # the gradient comes back in the caller's strides
    got = (float(layer.wavelength.grad), layer.radar_location.grad.cpu().numpy().astype(np.float64),
           xg.grad.cpu().numpy().astype(np.float64))
    # stage 1
    N, _, T, V, M = x.shape
    xc = xg.detach().contiguous()
    _, iq = layer.forward_debug(xg.detach())
    gz, _, _ = backward_gpu(xc, iq, go, edges, lam, loc, hop, _flags(mode), want_x=False)
    gz64, dz = check_stft_adjoint(tag, gz, iq, go, hop)
    # stage 2
    xn = xc.cpu().numpy()
    ref = ob.synth_adjoint(xn, gz64, edges, lam, loc, mode)
    delta = 2 * dz.reshape(N, -1).max(1)[:, None] * np.ones((N, T))
    prop = [ob.synth_adjoint(xn, np.stack((delta * (c == 0), delta * (c == 1)), -1), edges, lam, loc, mode) for c in (0, 1)]
    t_lam, t_loc, t_x = tolerances(ref, edges)
    tols = (t_lam + sum(_scale(p, "lam") for p in prop) + U32 * abs(ref["lam"]),
            t_loc + sum(_scale(p, "loc") for p in prop) + U32 * np.abs(ref["loc"]),
            t_x + sum(_scale(p, "x") for p in prop))
    errs, margins = compare(tag, got, ref, tols)
    low = {k: v for k, v in margins.items() if k.split("/")[0] != "phase" and v < 1}
    if low:     # the float32 dL/d(iq) hides this amplitude path here; the stage-level tests pin it
        print("  below the end-to-end tolerance (covered by the stage-level tests): %s" % low)
    return ref, got


@pytest.mark.gpu
@settings(max_examples=16, deadline=None, derandomize=True, suppress_health_check=[HealthCheck.too_slow, HealthCheck.data_too_large])
@given(sk=skeletons(star_cap=30), N=st.integers(1, 3), T=st.sampled_from([129, 130, 300, 777, 1500, 3001, 5000]),
       hop=st.sampled_from([8, 16, 37, 100, 300]), lam=st.sampled_from([5e-4, 1e-3, 5e-3]),
       loc=st.sampled_from([(0., 0., 0.), OFF_AXIS]), layout=st.sampled_from(["planar", "coordinate_innermost"]),
       seed=st.integers(0, 2 ** 16))
def test_module_backward_property(sk, N, T, hop, lam, loc, layout, seed):
    V, M, edges = sk
    if N * T * len(edges) * M > 1_500_000:
        N = 1
    x = _positions((N, 3, T, V, M), seed, layout=layout)
    check_module("V=%d M=%d E=%d N=%d T=%d hop=%d lam=%g %s" % (V, M, len(edges), N, T, hop, lam, layout),
                 x, edges, lam, loc, hop, seed)


# ---- GPU: edges -----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_absent_body_gives_exactly_zero():
    edges = [(0, 1), (1, 2), (2, 3), (0, 4), (4, 5), (5, 6), (0, 7), (7, 8), (8, 9), (9, 10), (3, 10), (6, 2)]
    x, giq, _ = _random_case((3, 3, 200, 11, 3), edges, 51)
    x[1, :, :, :, 2] = 0
    x[2, :, :, :, 0] = 0
    _, got = check_stage("absent body", x, giq, edges, 1e-3, OFF_AXIS, "seq")
    assert np.all(got[2][1, :, :, :, 2] == 0) and np.all(got[2][2, :, :, :, 0] == 0)
    assert np.abs(got[2][1, :, :, :, :2]).max() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["seq", "fma"])
def test_source_joint_at_the_radar(mode):
    """d = 0: the phase term is skipped (guard d > 0), the amplitude terms stay; the oracle defines the value."""
    loc = (0.3, -0.2, 1.5)
    edges = [(0, 1), (1, 2), (0, 3), (3, 4)]
    x, giq, _ = _random_case((2, 3, 150, 5, 2), edges, 52)
    x[0, :, 20:60, 0, 1] = torch.tensor(loc).view(3, 1)
    x[1, :, :, 3, 0] = torch.tensor(loc).view(3, 1)
    ref, _ = check_stage("source at the radar (%s)" % mode, x, giq, edges, 1e-3, loc, mode)
    d, _ = vro.range_phase_c(x[:, :, :, [0]], np.float32(loc), np.float32(1e-3), mode)
    assert int((d == 0).sum()) == 40


@pytest.mark.gpu
def test_bones_pointing_at_an_off_axis_radar():
    """Short bones on a ray from the radar: |u| -> 1, the amplitude's 1/c amplification, the u path large."""
    loc = np.array([0.3, -0.2, 1.5], np.float32)
    g = torch.Generator().manual_seed(53)
    N, T, V, M = 2, 200, 6, 2
    dirs = torch.randn(N, 3, T, 1, M, generator=g)
    dirs = dirs / dirs.norm(dim=1, keepdim=True)
    r = 0.8 + 0.01 * torch.arange(V, dtype=torch.float32).view(1, 1, 1, V, 1)
    x = (torch.from_numpy(loc).view(1, 3, 1, 1, 1) + dirs * r + 1e-4 * torch.randn(N, 3, T, V, M, generator=g)).float()
    edges = [(i, i + 1) for i in range(V - 1)]
    giq = torch.randn(N, T, 2, generator=g)
    ref, _ = check_stage("bones at the radar", x, giq, edges, 5e-3, tuple(loc), "seq")
    u_share = np.abs(ref["paths"]["u"]["x"]).max() / np.abs(ref["paths"]["phase"]["x"]).max()
    print("u path / phase path (max over entries) %.2e" % u_share)
    assert u_share > 1e-2


@pytest.mark.gpu
def test_128_bones_accepted_129_rejected():
    cabi = _lib()
    V, M, T = 34, 2, 200
    edges = [(i % V, (i * 7 + 3) % V if (i * 7 + 3) % V != i % V else (i + 1) % V) for i in range(128)]
    x, giq, _ = _random_case((2, 3, T, V, M), edges, 54)
    check_stage("E=128", x, giq, edges, 9e-4, OFF_AXIS, "seq")
    xg, iq = x.cuda(), torch.randn(2, T, 2, device="cuda")
    go = torch.randn(2, 256, T // 16 + 1, device="cuda")
    gz, gp, gx = backward_gpu(xg, iq, go, edges, 9e-4, OFF_AXIS, 16, 0)
    assert torch.isfinite(gp).all() and torch.isfinite(gx).all()
    bad = edges + [(0, 1)]
    with pytest.raises(NotImplementedError):
        synth_gpu(xg, giq, bad, 9e-4, OFF_AXIS, 0)
    with pytest.raises(NotImplementedError):
        backward_gpu(xg, iq, go, bad, 9e-4, OFF_AXIS, 16, 0)
    lam_t, loc_t = _params(9e-4, OFF_AXIS)
    src, dst = map(list, zip(*bad))
    gp = torch.zeros(4, dtype=torch.float64, device="cuda")
    rc = cabi.lib().vr_synth_adjoint_f32(xg.data_ptr(), giq.cuda().data_ptr(), 2, T, V, M, cabi.i32_array(src), cabi.i32_array(dst),
                                         129, lam_t.data_ptr(), loc_t.data_ptr(), 0, gp.data_ptr(), None, _stream())
    assert rc == cabi.VR_ERR_UNSUPPORTED


@pytest.mark.gpu
@pytest.mark.parametrize("T,hop", [(129, 16), (1000, 300)])
def test_shortest_sequence_and_uncovered_samples(T, hop):
    """T = 129 (the minimum) with hop 16; hop 300 > n_fft leaves samples no frame covers (dL/d(iq) = 0 there)."""
    edges = [(0, 1), (1, 2), (2, 3), (1, 4), (4, 5), (0, 6)]
    x = _positions((2, 3, T, 7, 3), 55)
    ref, _ = check_module("T=%d hop=%d" % (T, hop), x, edges, 1e-3, OFF_AXIS, hop, 56)
    if hop > 256:
        covered = np.zeros(T, bool)
        for f in range(T // hop + 1):
            covered[ob._reflect(f * hop - 128 + np.arange(256), T)] = True
        assert (~covered).sum() > 100


# ---- GPU: the grid-stride loops wrap -------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_grid_stride_wrap():
    """N from the SM count so that both kernels loop: N * F > 8 * 8 * SMs frames (adjoint STFT) and N * T > 16 * 128 * SMs
    steps (synthesis adjoint)."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    T, hop, V, M = 2100, 16, 11, 3
    F = T // hop + 1
    N = 2 * (16 * 128 * sms + T - 1) // T + 1
    assert N * F > 64 * sms and N * T > 2 * 2048 * sms
    print("SMs %d, N %d: %d frames, %d steps" % (sms, N, N * F, N * T))
    edges = [(0, 1), (1, 2), (2, 3), (3, 4), (1, 5), (5, 6), (6, 7), (0, 8), (8, 9), (9, 10), (5, 5 + 2), (2, 9)]
    lam, loc = 1e-3, OFF_AXIS
    g = torch.Generator(device="cuda").manual_seed(61)
    x = torch.randn(N, 3, T, V, M, device="cuda", generator=g) * 0.4
    go = torch.randn(N, 256, F, device="cuda", generator=g)
    layer = _layer(edges, lam, loc, hop)
    _, iq = layer.forward_debug(x)
    gz, gp_b, gx_b = backward_gpu(x, iq, go, edges, lam, loc, hop, 0)
    gp_s, gx_s = synth_gpu(x, gz, edges, lam, loc, 0)
    assert torch.equal(gx_s, gx_b)
    per_seq = []
    for n in range(N):
        gp_n, gx_n = synth_gpu(x[n:n + 1], gz[n:n + 1], edges, lam, loc, 0)
        assert torch.equal(gx_n[0], gx_b[n]), n
        per_seq.append(gp_n.cpu().numpy())
    per_seq = np.array(per_seq)
    d = np.abs(gp_s.cpu().numpy() - per_seq.sum(0)) / np.abs(per_seq).sum(0)
    print("batch parameters - sum over sequences: %s of the sum of |per-sequence gradient|" % d)
    assert np.all(d <= 1e-12), d
    for n in (0, N // 2, N - 1):                                # the adjoint STFT at both ends and the middle
        check_stft_adjoint("grid-stride n=%d" % n, gz[n:n + 1], iq[n:n + 1], go[n:n + 1], hop)
    for n in (0, N - 1):                                        # end to end from the GPU's own dL/d(iq)
        ref = ob.synth_adjoint(x[n:n + 1].cpu().numpy(), gz[n:n + 1].cpu().numpy(), edges, lam, loc, "seq")
        t_lam, t_loc, t_x = tolerances(ref, edges)
        got = (float(per_seq[n][0]), per_seq[n][1:], gx_b[n:n + 1].cpu().numpy().astype(np.float64))
        compare("grid-stride n=%d" % n, got, ref, (t_lam, t_loc, t_x))


# ---- GPU: the general-STFT route ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_general_stft_route():
    """train_stft_kernel=True (_SynthFunction): the module's gradients are vr_synth_adjoint_f32 fed the general STFT's own
    dL/d(iq) -- dL/dx bit for bit, the parameters within 1e-12 (and the float32 rounding of the module's result) -- and the
    oracle agrees with them."""
    edges = [(3, 0), (3, 1), (3, 2), (0, 4), (4, 5), (5, 6), (1, 7), (7, 8), (2, 8)]
    lam, loc, hop = 9e-4, OFF_AXIS, 16
    x = _positions((2, 3, 300, 9, 3), 71, layout="coordinate_innermost")
    layer = _layer(edges, lam, loc, hop, train_stft_kernel=True, train_wavelength=True, train_radar_location=True)
    xg = x.cuda().requires_grad_(True)
    out = layer(xg)
    go = torch.randn(out.shape, generator=torch.Generator().manual_seed(72)).cuda()
    (out * go).sum().backward()
    _, iq = layer.forward_debug(xg.detach())
    iq = iq.clone().requires_grad_(True)
    (layer.stft.logmag(iq) * go).sum().backward()
    gp, gx = synth_gpu(xg.detach(), iq.grad, edges, lam, loc, _lib().VR_FLAG_RANGE_FMA)
    assert xg.grad.stride() == xg.stride() and torch.equal(xg.grad, gx)
    gpn = gp.cpu().numpy()
    for got, want in ((float(layer.wavelength.grad), gpn[0]), *zip(layer.radar_location.grad.cpu().numpy(), gpn[1:])):
        assert abs(got - want) <= U32 * abs(want) + 1e-12 * abs(want), (got, want)
    ref = ob.synth_adjoint(x.contiguous().numpy(), iq.grad.cpu().numpy(), edges, lam, loc, "fma")
    compare("general STFT", (gpn[0], gpn[1:], gx.cpu().numpy().astype(np.float64)), ref, tolerances(ref, edges))


# ---- GPU: the up-sampled synthesis adjoint --------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("V,M,edges", [(7, 1, [(0, 1), (1, 2), (2, 3), (1, 4), (4, 5), (5, 6)]),
                                       (5, 3, [(2, 0), (2, 1), (2, 3), (2, 4), (0, 1), (0, 1)])])
def test_upsampled_synthesis_adjoint(V, M, edges):
    """vr_synth_adjoint_ups_kernel (positions from the spline's cubics) = vr_synth_adjoint_f32 on pad_frames(x) fed the same
    dL/d(iq), to 1e-12 of sum |term| -- beyond the NTU skeleton: other bone lists, M = 1 and 3, V * M not 50."""
    from skeleton_action_recognition_b200 import pad_frames
    from tests.test_upsampling_backward_gpu import _fused_backward
    T, k = 60, 10
    x = fx.s3_smooth(2, T=T, V=V, M=M).cuda()
    lam, loc = 1e-3, (0.3, -0.2, 1.5)
    layer = _layer(edges, lam, loc, 16)
    go = torch.randn(2, 256, k * T // 16 + 1, generator=torch.Generator().manual_seed(81)).cuda()
    _, iq, gz, gp = _fused_backward(layer, x, k, go)
    up = pad_frames(x, k, 3)
    assert torch.equal(iq, layer.forward_debug(up)[1])
    gp_ref, _ = synth_gpu(up, gz, edges, lam, loc, 0, want_x=False)
    ref = ob.synth_adjoint(up.cpu().numpy(), gz.cpu().numpy(), edges, lam, loc, "seq")
    a, b = gp.cpu().numpy(), gp_ref.cpu().numpy()
    t_lam, t_loc, _ = tolerances(ref, edges)
    print("ups vs materialised: lam %.2e loc %.2e of the tolerance" % (_ratio(a[0] - b[0], t_lam), _ratio(a[1:] - b[1:], t_loc)))
    assert _ratio(a[0] - b[0], t_lam) <= 1 and _ratio(a[1:] - b[1:], t_loc) <= 1, (a, b)
    assert _ratio(b[0] - ref["lam"], t_lam) <= 1 and _ratio(b[1:] - ref["loc"], t_loc) <= 1, (b, ref["lam"], ref["loc"])


# ---- GPU: NaN contract ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_parameter_gradient_is_nan_where_the_reference_is():
    """The input of test_aspect_cosine_beyond_one_gives_nan_like_the_reference: bones pointing exactly at the radar make the
    reference's u exceed 1 for some samples, its forward NaN there and, through the saved iq, the kernel's parameter gradient
    NaN.  Per sequence, the gradient is NaN exactly when the reference's float32 autograd gives NaN (today's behaviour)."""
    g = torch.Generator().manual_seed(3)
    N, T, V, M = 3, 800, 6, 2
    dirs = torch.randn(N, 3, T, 1, M, generator=g)
    dirs = dirs / dirs.norm(dim=1, keepdim=True)
    r = 12 + 30 * torch.rand(N, 1, T, 1, M, generator=g)
    radial = dirs * (r + torch.arange(V).float().view(1, 1, 1, V, 1) * 0.25)
    x = torch.randn(N, 3, T, V, M, generator=g) * 0.3 + 15
    x[0, :, 300:420] = radial[0, :, 300:420]
    x[2, :, :, :, 1] = radial[2, :, :, :, 1]
    edges = [(i, i + 1) for i in range(V - 1)]
    go = torch.randn(N, 256, T // 16 + 1, generator=g)
    nan_gpu, nan_ref = [], []
    for n in range(N):
        layer = _layer(edges, 1e-3, (0., 0., 0.), 16, train_wavelength=True, train_radar_location=True)
        (layer(x[n:n + 1].cuda()) * go[n:n + 1].cuda()).sum().backward()
        nan_gpu.append([bool(torch.isnan(layer.wavelength.grad)), *torch.isnan(layer.radar_location.grad).cpu().tolist()])
        a, b, _ = ob.autograd_grads(x[n:n + 1], go[n:n + 1].numpy(), edges=edges, wavelength=1e-3, dtype=torch.float32)
        nan_ref.append([bool(np.isnan(a)), *np.isnan(b).tolist()])
    print("NaN per sequence: kernel %s, reference %s" % (nan_gpu, nan_ref))
    assert nan_gpu == nan_ref
    assert all(nan_gpu[0]) and not any(nan_gpu[1]) and all(nan_gpu[2])
