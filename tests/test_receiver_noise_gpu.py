"""Receiver noise (C ABI VR_FLAG_NOISE + vr_set_noise, the `noise_std=` / `noise_seed=` keywords; DESIGN §3i): the forward
launches add xi[n, t] to the baseband z[n, t] of output n at step t before anything reads z.

  * The noise itself: a batch of all-zero skeletons has z = 0 exactly (zero-length bones have zero amplitude), so its I/Q
    IS xi.  It is checked against the numpy restatement below (Philox4x32-10 in uint64 arithmetic, Box-Muller in float64):
    the same bits except where float64 log / sincospi of the device and numpy round differently (at most 1e-6 of the
    values, and one float32 unit in the last place there), and against the normal distribution.
  * Every bitwise relation of the launch regimes holds with the noise on, and a noisy I/Q is the clean I/Q plus xi.
  * Gradients are those of the noisy spectrogram: oracle/backward.py's adjoint on the saved noisy I/Q.
The unmarked tests check the generator restatement, the C ABI's argument handling and the Python keywords without a GPU.

Shared helpers: the inputs (`_batch`, `_edges`, `_placements`: NTU-shaped batches, generic skeletons, per-sequence
placements with a |u| > 1 NaN sequence) and the NaN-aware bitwise comparison `_same` come from
tests/test_per_sequence_radar_gpu.py, and the two-stage gradient check (`backward_gpu`, `check_stft_adjoint`, `tolerances`,
`compare`) from tests/test_backward_property_gpu.py, so that the noisy routes are held to exactly the inputs and tolerances
the noiseless ones are."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import backward as ob
from oracle import virtual_radar_oracle as vro
from tests.test_per_sequence_radar_gpu import _batch, _edges, _placements, _same

SEEDS = (0, 2 ** 64 - 1, 0x9E3779B97F4A7C15)
LOC0 = (1.0, 2.0, 3.0)          # placement of the all-zero batches (any placement gives z = 0 there)


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


# ---- the numpy restatement of the definition ----------------------------------------------------------------------------------
_M32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Random123's philox4x32-10 on uint64 arrays holding 32-bit words -> (w0, w1, w2, w3)."""
    c0, c1, c2, c3 = [np.asarray(v, np.uint64) & _M32 for v in (c0, c1, c2, c3)]
    k0, k1 = np.asarray(k0, np.uint64) & _M32, np.asarray(k1, np.uint64) & _M32
    for r in range(10):
        if r:
            k0, k1 = (k0 + np.uint64(0x9E3779B9)) & _M32, (k1 + np.uint64(0xBB67AE85)) & _M32
        p0, p1 = np.uint64(0xD2511F53) * c0, np.uint64(0xCD9E8D57) * c2      # 32 x 32 -> 64 bits, exact in uint64
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & _M32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & _M32
    return c0, c1, c2, c3


def _sincospi(x):
    """(sin(pi x), cos(pi x)) in float64 with an exact reduction to |r| <= 1/4 (x = q / 2 + r, x a multiple of 2^-52)."""
    q = np.rint(x * 2.0)
    a = np.pi * (x - q * 0.5)
    s0, c0 = np.sin(a), np.cos(a)
    qi = q.astype(np.int64) & 3
    return np.choose(qi, [s0, c0, -s0, -c0]), np.choose(qi, [c0, -s0, -c0, s0])


def xi_ref(seed, n, t, sigma):
    """xi[n, t] (broadcast over n, t and sigma) -> (I, Q) float32."""
    n, t = np.asarray(n, np.uint64), np.asarray(t, np.uint64)
    seed = int(seed)
    w0, w1, w2, w3 = philox4x32_10(t & _M32, t >> np.uint64(32), n & _M32, n >> np.uint64(32), seed & 0xFFFFFFFF, seed >> 32)
    u1 = ((((w1 << np.uint64(32)) | w0) >> np.uint64(11)) + np.uint64(1)).astype(np.float64) * 2.0 ** -53
    u2 = (((w3 << np.uint64(32)) | w2) >> np.uint64(11)).astype(np.float64) * 2.0 ** -53
    s, c = _sincospi(2.0 * u2)
    a = np.asarray(sigma, np.float32).astype(np.float64) * np.sqrt(0.5) * np.sqrt(-2.0 * np.log(u1))
    return (a * c).astype(np.float32), (a * s).astype(np.float32)


def _assert_bits(got, want):
    """The same float32 values on at least 1 - 1e-6 of them, one unit in the last place apart elsewhere."""
    got, want = np.asarray(got, np.float32), np.asarray(want, np.float32)
    assert np.isfinite(got).all()
    diff = got != want
    assert diff.sum() <= 1e-6 * got.size, (int(diff.sum()), got.size)
    ulp = np.spacing(np.maximum(np.abs(got), np.abs(want)))
    assert (np.abs(got.astype(np.float64) - want) <= ulp).all()


def test_philox_known_answers():
    """Random123's known-answer vectors for philox4x32-10 (kat_vectors)."""
    for ctr, key, want in (((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
                           ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
                           ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
                            (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))):
        assert tuple(int(w) for w in philox4x32_10(*ctr, *key)) == want


def test_reference_transform():
    """The reference's uniforms stay inside (0, 1] and [0, 1), and its sincospi agrees with numpy's sin / cos."""
    x = np.random.default_rng(0).integers(0, 2 ** 53, 100_000).astype(np.float64) * 2.0 ** -52
    s, c = _sincospi(x)
    assert np.allclose(s, np.sin(np.pi * x), atol=1e-15) and np.allclose(c, np.cos(np.pi * x), atol=1e-15)
    i, q = xi_ref(5, np.arange(1000)[:, None], np.arange(100)[None, :], np.float32(2.0))
    assert np.isfinite(i).all() and np.isfinite(q).all()
    assert abs(float(np.mean(i.astype(np.float64) ** 2 + q.astype(np.float64) ** 2)) - 4.0) < 0.1


# ---- launches -----------------------------------------------------------------------------------------------------------------
def _seed_tensor(seed):
    return torch.tensor(seed - 2 ** 64 if seed >= 2 ** 63 else seed, dtype=torch.int64, device="cuda")


def _zero_noise(entry, N, T, std, seed, k=None):
    """The I/Q of N all-zero sequences through one C-ABI entry with VR_FLAG_NOISE: xi itself.  entry: "debug"
    (vr_forward_debug_f32), "synth" (vr_synth_f32) or "synth_upsampled" (vr_synth_upsampled_f32, T raw frames, k = the
    factor) -> (N, T or k T, 2) on the GPU."""
    cabi = _cabi()
    L = cabi.lib()
    src, dst = map(list, zip(*vro.NTU_EDGES))
    sc, dc = cabi.i32_array(src), cabi.i32_array(dst)
    x = torch.zeros(N, 3, T, 25, 2, device="cuda")
    lam = torch.full((N,), 1e-3, device="cuda")
    loc = torch.tensor(LOC0, device="cuda").expand(N, 3).contiguous()
    std = std.cuda().contiguous()
    seed_t = _seed_tensor(seed)
    flags = cabi.VR_FLAG_PER_SEQUENCE | cabi.VR_FLAG_NOISE
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    iq = torch.empty(N, T * (k or 1), 2, device="cuda")
    cabi.set_noise(std, seed_t)
    if entry == "debug":
        out = torch.empty(N, 256, T // 16 + 1, device="cuda")
        rc = L.vr_forward_debug_f32(x.data_ptr(), N, T, 25, 2, sc, dc, len(src), lam.data_ptr(), loc.data_ptr(), 256, 16,
                                    flags, out.data_ptr(), iq.data_ptr(), st)
    elif entry == "synth":
        rc = L.vr_synth_f32(x.data_ptr(), N, T, 25, 2, sc, dc, len(src), lam.data_ptr(), loc.data_ptr(), flags, iq.data_ptr(), st)
    else:
        nbytes = int(L.vr_upsampled_workspace_bytes(N, T, 25, 2))
        work = torch.empty(nbytes // 8 + 1, dtype=torch.float64, device="cuda")
        rc = L.vr_synth_upsampled_f32(x.data_ptr(), N, T, 25, 2, sc, dc, len(src), lam.data_ptr(), loc.data_ptr(), flags, k,
                                      ctypes.c_float(3.0), work.data_ptr(), nbytes, iq.data_ptr(), st)
    cabi.check(rc)
    torch.cuda.synchronize()
    return iq


def _std(N, zero_every=None):
    s = 0.5 + 0.25 * (torch.arange(N) % 7).float()
    if zero_every:
        s[::zero_every] = 0.0
    return s


# ---- 1. the noise itself ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("seed", SEEDS)
@pytest.mark.parametrize("shape", [(3000, 300), (2, 75000)])      # (outputs, steps): n to a few thousand, t to 75 000
@pytest.mark.parametrize("entry", ["debug", "synth"])
def test_zero_batch_iq_is_the_reference_noise(entry, shape, seed):
    N, T = shape
    std = _std(N)
    iq = _zero_noise(entry, N, T, std, seed).cpu().numpy()
    i, q = xi_ref(seed, np.arange(N)[:, None], np.arange(T)[None, :], std.numpy()[:, None])
    _assert_bits(iq[..., 0], i)
    _assert_bits(iq[..., 1], q)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", SEEDS)
def test_zero_batch_upsampled_noise_is_keyed_by_the_upsampled_step(seed):
    N, T, k = 3, 300, 250
    std = _std(N)
    iq = _zero_noise("synth_upsampled", N, T, std, seed, k=k).cpu().numpy()
    i, q = xi_ref(seed, np.arange(N)[:, None], np.arange(k * T)[None, :], std.numpy()[:, None])
    _assert_bits(iq[..., 0], i)
    _assert_bits(iq[..., 1], q)


@pytest.mark.gpu
def test_noise_statistics():
    """10^7 samples of one fixed seed: mean, per-component variance sigma^2 / 2, correlations of I with Q and of
    neighbouring steps and outputs, and a Kolmogorov-Smirnov test against the normal distribution."""
    from scipy import stats
    N, T, sigma = 1000, 5000, 1.5
    iq = _zero_noise("synth", N, T, torch.full((N,), sigma), 12345).cpu().numpy().astype(np.float64)
    var = sigma ** 2 / 2
    for c in (0, 1):
        v = iq[..., c]
        cnt = v.size
        assert abs(v.mean()) <= 5 * np.sqrt(var / cnt), v.mean()
        # the variance of a sample variance of a normal: 2 var^2 / count
        assert abs(v.var() - var) <= 5 * var * np.sqrt(2.0 / cnt), v.var()
        for a, b in ((v[:, 1:], v[:, :-1]), (v[1:], v[:-1])):        # neighbouring t, neighbouring n
            r = np.corrcoef(a.ravel(), b.ravel())[0, 1]
            assert abs(r) <= 5 / np.sqrt(a.size), r
        p = stats.kstest(v.ravel() / np.sqrt(var), "norm").pvalue
        assert p > 1e-4, p
    r = np.corrcoef(iq[..., 0].ravel(), iq[..., 1].ravel())[0, 1]
    assert abs(r) <= 5 / np.sqrt(N * T), r


# ---- 2. the bitwise relations with the noise on -------------------------------------------------------------------------------
def _noise_kw(N, seed=77, zero_every=None):
    return dict(noise_std=_std(N, zero_every).cuda(), noise_seed=seed)


CASES = {                     # (N, T, V, M, layout)
    "ntu": (5, 300, 25, 2, "planar"),
    "coordinate_innermost": (4, 300, 25, 2, "coordinate_innermost"),
    "one_body": (4, 300, 25, 1, "planar"),
    "three_bodies": (3, 300, 25, 3, "planar"),
    "generic_vm": (4, 256, 17, 2, "planar"),
    "long_park": (2, 5000, 25, 2, "planar"),
    "ntu_many_jobs": (1300, 300, 25, 2, "planar"),      # every CTA and team runs several jobs
    "park_many_jobs": (100, 5000, 25, 2, "planar"),     # several jobs per sequence: their halos overlap
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("mode", [0, 1, "ready"])
def test_noisy_iq_is_clean_iq_plus_noise_in_every_regime(case, mode, schedule):
    """The debug launch's noisy I/Q is its clean I/Q + xi (float32, on the GPU), the |u| > 1 NaN mask is unchanged, and the
    spectrogram of each schedule (cooperative, team jobs, inputs-ready) is the debug launch's bits."""
    cabi = _cabi()
    N, T, V, M, layout = CASES[case]
    if case == "park_many_jobs":
        src, dst = map(list, zip(*vro.NTU_EDGES))
        assert cabi.plan(N, T, V, M, src, dst)["jobs_per_seq"] > 1
    nan_seq = 1 if V == 25 and N < 1000 else None
    x = _batch(N, T, V, M, seed=3, layout=layout, nan_seq=nan_seq).cuda()
    lam, loc = [t.cuda() for t in _placements(N, seed=2, nan_seq=nan_seq)]
    kw = _noise_kw(N)
    layer = _layer(edges=_edges(V))
    with torch.no_grad():
        xc, flags = layer._prepare(x)
        pl = layer._placements(x, loc, lam, **kw)
        noisy_out, noisy = layer._launch(xc, flags | pl[2], want_iq=True, lam=pl[0], loc=pl[1], noise=pl[3])
        clean_out, clean = layer._launch(xc, flags | cabi.VR_FLAG_PER_SEQUENCE, want_iq=True, lam=lam, loc=loc)
        xi = _zero_noise("debug", N, T, kw["noise_std"], kw["noise_seed"])
        assert _same(noisy, clean + xi)
        assert torch.equal(torch.isnan(noisy_out), torch.isnan(clean_out))
        if nan_seq is not None:
            assert torch.isnan(noisy_out[nan_seq]).any()
        schedule(mode if mode != "ready" else -1)
        layer.assume_inputs_ready = mode == "ready"
        out = layer(x, radar_location=loc, wavelength=lam, **kw)
    assert _same(out, noisy_out)
    assert not torch.equal(torch.nan_to_num(out), torch.nan_to_num(clean_out))


@pytest.mark.gpu
@pytest.mark.parametrize("T", [300, 6000])            # F = 19 <= 256 columns, F = 376 > 256 (only kept frames)
@pytest.mark.parametrize("image_size", [256, 64])
def test_forward_image_is_the_resized_noisy_spectrogram(T, image_size):
    x = _batch(4, T, seed=4).cuda()
    lam, loc = [t.cuda() for t in _placements(4, seed=1)]
    layer = _layer()
    with torch.no_grad():
        img = layer.forward_image(x, image_size, radar_location=loc, wavelength=lam, **_noise_kw(4))
        ref = torch.nn.functional.interpolate(layer(x, radar_location=loc, wavelength=lam, **_noise_kw(4)).unsqueeze(1),
                                              image_size)
    assert torch.equal(img, ref)


@pytest.mark.gpu
@pytest.mark.parametrize("image_size", [None, 64])
@pytest.mark.parametrize("stft", ["fused", "general"])
def test_forward_upsampled_is_forward_of_the_padded_batch(image_size, stft):
    from skeleton_action_recognition_b200 import pad_frames
    x = _batch(3, 24, seed=5).cuda()
    lam, loc = [t.cuda() for t in _placements(3, seed=2)]
    layer = _layer(**(dict(train_stft_kernel=True) if stft == "general" else {}))
    with torch.no_grad():
        out = layer.forward_upsampled(x, 40, 3, image_size, radar_location=loc, wavelength=lam, **_noise_kw(3))
        xp = pad_frames(x, 40, 3)
        if image_size is None:
            ref = layer(xp, radar_location=loc, wavelength=lam, **_noise_kw(3))
        else:
            ref = layer.forward_image(xp, image_size, radar_location=loc, wavelength=lam, **_noise_kw(3))
    assert torch.equal(out, ref)


@pytest.mark.gpu
@pytest.mark.parametrize("R", [1, 2, 3, 7])
@pytest.mark.parametrize("route", ["forward", "image", "upsampled"])
def test_views_equal_the_repeated_batch(route, R):
    N = 3
    T = 24 if route == "upsampled" else 300
    x = _batch(N, T, seed=6).cuda()
    g = np.random.default_rng(R)
    loc = torch.from_numpy((g.normal(size=(N, R, 3)) * 1.5).astype(np.float32)).cuda()
    lam = torch.full((N, R), 1e-3, device="cuda")
    std = _std(N * R, zero_every=4).cuda()
    kw = dict(image_size=64) if route == "image" else dict(num_pad_frames=20) if route == "upsampled" else {}
    layer = _layer()
    with torch.no_grad():
        out = layer.forward_views(x, loc, lam, noise_std=std.view(N, R), noise_seed=5, **kw)
        rkw = dict(radar_location=loc.reshape(N * R, 3), wavelength=lam.reshape(N * R), noise_std=std, noise_seed=5)
        xr = x.repeat_interleave(R, 0)
        if route == "image":
            ref = layer.forward_image(xr, 64, **rkw)
        elif route == "upsampled":
            ref = layer.forward_upsampled(xr, 20, 3, **rkw)
        else:
            ref = layer(xr, **rkw)
    assert torch.equal(out.reshape(ref.shape), ref)


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft", [128, 256, 512])
def test_general_stft_reads_the_noisy_iq(n_fft):
    """The general-kernel route (vr_synth_f32 with the noise, then the tcgen05 STFT) reads the fused debug launch's noisy
    I/Q bit for bit."""
    cabi = _cabi()
    x = _batch(4, 600, seed=6).cuda()
    lam, loc = [t.cuda() for t in _placements(4, seed=3)]
    layer = _layer(n_fft=n_fft, train_stft_kernel=True)
    kw = _noise_kw(4)
    with torch.no_grad():
        out = layer(x, radar_location=loc, wavelength=lam, **kw)
        pl = layer._placements(x, loc, lam, **kw)
        _, iq = layer._launch(x.contiguous(), pl[2], want_iq=True, lam=pl[0], loc=pl[1], noise=pl[3])
        ref = layer.stft.logmag(iq)
    assert pl[2] & cabi.VR_FLAG_NOISE
    assert torch.equal(out, ref)


@pytest.mark.gpu
@pytest.mark.parametrize("route", ["forward", "image", "upsampled", "general"])
def test_zero_noise_level_is_the_noiseless_spectrogram(route):
    """sigma = 0 everywhere is the noiseless spectrogram (compared as spectrograms: -0 + 0 = +0 in the I/Q); sigma = 0 next
    to noisy outputs in one launch leaves exactly those outputs noiseless."""
    N = 6
    T = 24 if route == "upsampled" else 300
    x = _batch(N, T, seed=9).cuda()
    lam, loc = [t.cuda() for t in _placements(N, seed=5)]
    layer = _layer(**(dict(train_stft_kernel=True) if route == "general" else {}))

    def run(**kw):
        if route == "image":
            return layer.forward_image(x, 64, radar_location=loc, wavelength=lam, **kw)
        if route == "upsampled":
            return layer.forward_upsampled(x, 20, 3, radar_location=loc, wavelength=lam, **kw)
        return layer(x, radar_location=loc, wavelength=lam, **kw)
    with torch.no_grad():
        clean = run()
        assert torch.equal(run(noise_std=0.0, noise_seed=3), clean)
        mixed = run(**_noise_kw(N, seed=3, zero_every=2))
    for n in range(N):
        assert torch.equal(mixed[n], clean[n]) == (n % 2 == 0), n


@pytest.mark.gpu
def test_noise_is_deterministic_across_calls_streams_and_graph_replays():
    N, T = 8, 300
    x = _batch(N, T, seed=10).cuda()
    layer = _layer()
    std = _std(N).cuda()
    seed = torch.tensor(11, dtype=torch.int64, device="cuda")
    with torch.no_grad():
        first = layer(x, noise_std=std, noise_seed=seed)
        assert torch.equal(layer(x, noise_std=std, noise_seed=11), first)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            other = layer(x, noise_std=std, noise_seed=seed)
        torch.cuda.current_stream().wait_stream(s)
        assert torch.equal(other, first)
        # a different seed changes every output
        second = layer(x, noise_std=std, noise_seed=2 ** 64 - 1)
        for n in range(N):
            assert not torch.equal(second[n], first[n]), n
        # CUDA graph: the seed tensor is read at replay time
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            layer(x, noise_std=std, noise_seed=seed)               # warm-up on the capture stream
        torch.cuda.current_stream().wait_stream(s)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            captured = layer(x, noise_std=std, noise_seed=seed)
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(captured, first)
        seed.fill_(-1)                                              # the bits of 2^64 - 1
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(captured, second)
        # without a seed every call draws one from torch's CUDA generator: reproducible under torch.manual_seed
        torch.manual_seed(4)
        a = layer(x, noise_std=std)
        b = layer(x, noise_std=std)
        torch.manual_seed(4)
        assert torch.equal(layer(x, noise_std=std), a) and not torch.equal(a, b)


@pytest.mark.gpu
def test_noisy_spectrogram_meets_the_parity_criterion():
    """The fused spectrogram with noise against the oracle's STFT of the same noisy I/Q (float64 oracle kernels)."""
    x = _batch(3, 300, seed=12).cuda()
    lam, loc = [t.cuda() for t in _placements(3, seed=8)]
    layer = _layer()
    kw = _noise_kw(3)
    with torch.no_grad():
        pl = layer._placements(x, loc, lam, **kw)
        out, iq = layer._launch(x.contiguous(), pl[2], want_iq=True, lam=pl[0], loc=pl[1], noise=pl[3])
    o = vro.OracleVirtualRadar(dtype=torch.float64)
    ref = vro.stft_logmag(iq.cpu().double(), o.stft, 256)
    rep = vro.parity_report(out.cpu().numpy(), ref.numpy())
    assert vro.parity_ok(rep), rep


# ---- 3. gradients -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["planar", "coordinate_innermost"])
def test_gradients_are_those_of_the_noisy_spectrogram(layout):
    """Per-sequence placement and x gradients with the noise on, in the two stages of tests/test_backward_property_gpu.py's
    check_module: dL/d(iq) of the saved noisy I/Q against ob.stft_adjoint (the oracle's graph with xi added to its I/Q),
    then the gradients against ob.synth_adjoint of that float64 dL/d(iq), with that file's tolerances."""
    from tests.test_backward_property_gpu import (U32, _scale, backward_gpu, check_stft_adjoint, compare, tolerances)
    N, T = 2, 300
    x = _batch(N, T, seed=13, layout=layout)
    mode = vro.distance_mode_for(x)
    lam = torch.tensor([1e-3, 5e-4])
    loc = torch.tensor([[0.5, -1.0, 2.0], [0.0, 0.0, 0.0]])
    layer = _layer()
    kw = dict(noise_std=torch.tensor([0.3, 1.0], device="cuda"), noise_seed=21)
    xg = x.cuda().requires_grad_(True)
    lam_t, loc_t = lam.cuda().requires_grad_(True), loc.cuda().requires_grad_(True)
    out = layer(xg, radar_location=loc_t, wavelength=lam_t, **kw)
    go = torch.randn(out.shape, generator=torch.Generator().manual_seed(1)).cuda()
    (out * go).sum().backward()
    xc = xg.detach().contiguous()
    flags = _cabi().VR_FLAG_RANGE_FMA if mode == "fma" else 0
    with torch.no_grad():
        pl = layer._placements(xc, loc_t.detach(), lam_t.detach(), **kw)
        _, iq = layer._launch(xc, flags | pl[2], want_iq=True, lam=pl[0], loc=pl[1], noise=pl[3])
    for n in range(N):
        ln, Ln = float(lam[n]), tuple(loc[n].tolist())
        gz, _, _ = backward_gpu(xc[n:n + 1], iq[n:n + 1].contiguous(), go[n:n + 1].contiguous(), vro.NTU_EDGES, ln, Ln,
                                16, flags, want_x=False)
        gz64, dz = check_stft_adjoint("noise n=%d" % n, gz, iq[n:n + 1], go[n:n + 1], 16)
        xn = xc[n:n + 1].cpu().numpy()
        ref = ob.synth_adjoint(xn, gz64, vro.NTU_EDGES, ln, Ln, mode)
        delta = 2 * dz.max() * np.ones((1, T))
        prop = [ob.synth_adjoint(xn, np.stack((delta * (c == 0), delta * (c == 1)), -1), vro.NTU_EDGES, ln, Ln, mode)
                for c in (0, 1)]
        t_lam, t_loc, t_x = tolerances(ref, vro.NTU_EDGES)
        tols = (t_lam + sum(_scale(p, "lam") for p in prop) + U32 * abs(ref["lam"]),
                t_loc + sum(_scale(p, "loc") for p in prop) + U32 * np.abs(ref["loc"]),
                t_x + sum(_scale(p, "x") for p in prop))
        got = (float(lam_t.grad[n]), loc_t.grad[n].cpu().numpy().astype(np.float64),
               xg.grad[n:n + 1].cpu().numpy().astype(np.float64))
        compare("noise %s n=%d" % (layout, n), got, ref, tols)


def _grads(route, x, lam, loc, std, seed):
    layer = _layer(**(dict(train_stft_kernel=True) if route == "general" else {}))
    lam_t, loc_t = lam.cuda().requires_grad_(True), loc.cuda().requires_grad_(True)
    xg = x.cuda().requires_grad_(route != "upsampled")
    kw = dict(radar_location=loc_t, wavelength=lam_t, noise_std=std.cuda(), noise_seed=seed)
    out = layer.forward_upsampled(xg, 20, 3, **kw) if route == "upsampled" else layer(xg, **kw)
    w = torch.cos(torch.arange(out[0].numel(), device=out.device, dtype=torch.float32) * 0.37).view(out.shape[1:])
    (out * w).sum().backward()
    torch.cuda.synchronize()
    return lam_t.grad, loc_t.grad, xg.grad


@pytest.mark.gpu
@pytest.mark.parametrize("route", ["fused", "general", "upsampled"])
def test_noisy_gradients_depend_only_on_the_sequence_and_its_position(route):
    """For a fixed (seed, n) output n's gradients are the same bits whatever the other sequences of the batch and the
    batch size; the noise makes them differ from the noiseless ones."""
    N = 5
    T = 24 if route == "upsampled" else 300
    x = _batch(N, T, seed=14)
    lam, loc = _placements(N, seed=4)
    std = _std(N)
    gl, gL, gx = _grads(route, x, lam, loc, std, 9)
    x2 = x.clone()
    x2[3:] = _batch(N - 3, T, seed=15)                  # other sequences after position 2
    l2, L2, g2 = _grads(route, x2, lam, loc, std, 9)
    assert torch.equal(l2[:3], gl[:3]) and torch.equal(L2[:3], gL[:3])
    s3 = _grads(route, x[:3], lam[:3], loc[:3], std[:3], 9)
    assert torch.equal(s3[0], gl[:3]) and torch.equal(s3[1], gL[:3])
    if gx is not None:
        assert torch.equal(g2[:3], gx[:3]) and torch.equal(s3[2], gx[:3])
    quiet = _grads(route, x, lam, loc, torch.zeros(N), 9)
    assert not torch.equal(quiet[1], gL)
    again = _grads(route, x, lam, loc, std, 9)
    assert torch.equal(again[0], gl) and torch.equal(again[1], gL)


# ---- 4. errors ----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_bad_noise_keywords_raise_on_the_gpu():
    layer = _layer()
    x = _batch(4, 300).cuda()
    with pytest.raises(ValueError):
        layer(x, noise_std=torch.ones(3, device="cuda"))                       # does not broadcast to (4,)
    with pytest.raises(ValueError):
        layer.forward_views(x, torch.zeros(2, 3, device="cuda"), noise_std=torch.ones(4, 3, device="cuda"))
    with pytest.raises(RuntimeError):
        layer(x, noise_std=torch.ones(4))                                      # CPU tensor
    with pytest.raises(RuntimeError):
        layer(x, noise_std=1.0, noise_seed=torch.tensor(3))                    # CPU seed
    with pytest.raises(ValueError):
        layer(x, noise_std=torch.ones(4, device="cuda", requires_grad=True))
    # the keywords reach the layer through Model
    from skeleton_action_recognition_b200.models.resnet import Model
    model = Model(num_classes=5, num_filters=8, image_size=64, device="cuda").cuda().eval()
    with torch.no_grad():
        a = model.spectrogram_image(x, noise_std=0.5, noise_seed=1)
        assert torch.equal(a, model.virtual_radar.forward_image(x, 64, noise_std=0.5, noise_seed=1))
        assert model(x, noise_std=0.5, noise_seed=1).shape == (4, 5)


def test_python_rejects_bad_noise_keywords():
    """Checked before anything reaches a device."""
    from skeleton_action_recognition_b200 import VirtualRadar
    x = torch.zeros(4, 3, 300, 25, 2)
    bad = [dict(noise_std=torch.ones(4, requires_grad=True)),
           dict(noise_std=torch.ones(4, dtype=torch.float64)),
           dict(noise_std=torch.ones(4, dtype=torch.float16)),
           dict(noise_std=-1.0), dict(noise_std=float("nan")), dict(noise_std=float("inf")), dict(noise_std=True),
           dict(noise_std="1"),
           dict(noise_std=1.0, noise_seed=1.5), dict(noise_std=1.0, noise_seed=-1), dict(noise_std=1.0, noise_seed=2 ** 64),
           dict(noise_std=1.0, noise_seed=True),
           dict(noise_std=1.0, noise_seed=torch.tensor([3])),
           dict(noise_std=1.0, noise_seed=torch.tensor(3, dtype=torch.int32)),
           dict(noise_std=1.0, noise_seed=torch.tensor(3.0)),
           dict(noise_seed=3)]
    for kw in bad:
        with pytest.raises(ValueError):
            VirtualRadar._noise(x, kw.get("noise_std"), kw.get("noise_seed"), (4,))
    assert VirtualRadar._noise(x, None, None, (4,)) is None
    std, seed = VirtualRadar._noise(x, 0.25, 2 ** 64 - 1, (4, 3))
    assert std.shape == (12,) and std.dtype == torch.float32 and bool((std == 0.25).all())
    assert seed.dtype == torch.int64 and seed.dim() == 0 and int(seed) == -1
    assert int(VirtualRadar._noise(x, 1.0, 2 ** 63 - 1, (4,))[1]) == 2 ** 63 - 1
    assert int(VirtualRadar._noise(x, 1.0, 2 ** 63, (4,))[1]) == -2 ** 63


def test_cabi_rejects_bad_noise():
    cabi = _cabi()
    L = cabi.lib()
    src, dst = map(list, zip(*vro.NTU_EDGES))
    sc, dc = cabi.i32_array(src), cabi.i32_array(dst)
    ps, nz = cabi.VR_FLAG_PER_SEQUENCE, cabi.VR_FLAG_NOISE
    fake = ctypes.c_void_p(256)                     # never dereferenced: the checks come first
    args = lambda flags, lam=fake: (fake, 4, 300, 25, 2, sc, dc, len(src), lam, fake, 256, 16, flags, fake, None)   # noqa: E731
    assert cabi.VR_FLAG_NOISE == 8
    # null pointers
    assert L.vr_set_noise(None, fake) == cabi.VR_ERR_ARG
    assert L.vr_set_noise(fake, None) == cabi.VR_ERR_ARG
    assert L.vr_set_noise(fake, ctypes.c_void_p(260)) == cabi.VR_ERR_ARG           # seed not 8-byte aligned
    # the flag without a pending setting (the failed setters above left none)
    assert L.vr_forward_f32(*args(ps | nz)) == cabi.VR_ERR_ARG
    assert "vr_set_noise" in cabi.last_error()
    # the flag without VR_FLAG_PER_SEQUENCE: rejected, and the setting is consumed
    assert L.vr_set_noise(fake, fake) == cabi.VR_OK
    assert L.vr_forward_f32(*args(nz)) == cabi.VR_ERR_ARG
    assert "VR_FLAG_PER_SEQUENCE" in cabi.last_error()
    assert L.vr_forward_f32(*args(ps | nz)) == cabi.VR_ERR_ARG
    assert "vr_set_noise" in cabi.last_error()
    # a call that fails for another reason consumes it too, in every entry that takes the flag
    entries = [
        lambda f: L.vr_forward_f32(*args(f, lam=None)),
        lambda f: L.vr_forward_debug_f32(fake, 4, 300, 25, 2, sc, dc, len(src), None, fake, 256, 16, f, fake, fake, None),
        lambda f: L.vr_forward_image_f32(fake, 4, 300, 25, 2, sc, dc, len(src), None, fake, 256, 16, f, 64, fake, None),
        lambda f: L.vr_synth_f32(fake, 4, 300, 25, 2, sc, dc, len(src), None, fake, f, fake, None),
        lambda f: L.vr_forward_upsampled_f32(fake, 4, 24, 25, 2, sc, dc, len(src), None, fake, 256, 16, f, 10,
                                             ctypes.c_float(3.0), 0, fake, 1 << 30, fake, None),
        lambda f: L.vr_forward_upsampled_debug_f32(fake, 4, 24, 25, 2, sc, dc, len(src), None, fake, 256, 16, f, 10,
                                                   ctypes.c_float(3.0), fake, 1 << 30, fake, fake, None),
        lambda f: L.vr_synth_upsampled_f32(fake, 4, 24, 25, 2, sc, dc, len(src), None, fake, f, 10, ctypes.c_float(3.0),
                                           fake, 1 << 30, fake, None),
    ]
    for i, call in enumerate(entries):
        assert L.vr_set_noise(fake, fake) == cabi.VR_OK
        assert call(ps | nz) == cabi.VR_ERR_ARG, i
        assert "must not be null" in cabi.last_error(), (i, cabi.last_error())
        assert L.vr_forward_f32(*args(ps | nz)) == cabi.VR_ERR_ARG, i
        assert "vr_set_noise" in cabi.last_error(), i
    # the host entry and the backward entries do not take the flag
    x = np.zeros((1, 3, 300, 25, 2), np.float32)
    out = np.zeros((1, 256, 19), np.float32)
    hloc = (ctypes.c_float * 3)(0, 0, 0)
    rejecting = [
        (lambda f: L.vr_forward_host_f32(x.ctypes.data, 1, 300, 25, 2, sc, dc, len(src), ctypes.c_float(1e-3), hloc, 256, 16,
                                         f, out.ctypes.data, 0), "VR_FLAG_NOISE"),
        (lambda f: L.vr_backward_f32(fake, fake, fake, 4, 300, 25, 2, sc, dc, len(src), fake, fake, 256, 16, f, fake, fake,
                                     None, None), "unknown flags"),
        (lambda f: L.vr_backward_params_f32(fake, fake, fake, 4, 300, 25, 2, sc, dc, len(src), fake, fake, 256, 16, f, fake,
                                            fake, None), "unknown flags"),
        (lambda f: L.vr_synth_adjoint_f32(fake, fake, 4, 300, 25, 2, sc, dc, len(src), fake, fake, f, fake, None, None),
         "unknown flags"),
        (lambda f: L.vr_backward_upsampled_params_f32(fake, fake, fake, 4, 24, 25, 2, sc, dc, len(src), fake, fake, 256, 16,
                                                      f, 10, fake, fake, None), "unknown flags"),
        (lambda f: L.vr_synth_adjoint_upsampled_f32(fake, fake, 4, 24, 25, 2, sc, dc, len(src), fake, fake, f, 10, fake,
                                                    None), "unknown flags"),
    ]
    for i, (call, msg) in enumerate(rejecting):
        for flags in (nz, ps | nz):
            assert L.vr_set_noise(fake, fake) == cabi.VR_OK
            assert call(flags) == cabi.VR_ERR_ARG, (i, flags)
            assert msg in cabi.last_error(), (i, cabi.last_error())
            # the rejected call consumed the setting: it cannot reach the next launch
            assert L.vr_forward_f32(*args(ps | nz)) == cabi.VR_ERR_ARG, i
            assert "vr_set_noise" in cabi.last_error(), i
    # a call without the flag leaves the setting pending
    assert L.vr_set_noise(fake, fake) == cabi.VR_OK
    assert L.vr_backward_f32(fake, fake, fake, 4, 300, 25, 2, sc, dc, len(src), fake, fake, 256, 16, 1 << 20, fake, fake,
                             None, None) == cabi.VR_ERR_ARG
    assert L.vr_forward_f32(*args(ps | nz, lam=None)) == cabi.VR_ERR_ARG
    assert "must not be null" in cabi.last_error()
