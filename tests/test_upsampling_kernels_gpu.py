"""The temporal up-sampling kernels (csrc/vr_pad_frames.cuh and the fused evaluation of csrc/vr_kernels.cuh) against a
long-double spline oracle, in every launch regime.

scipy is exact only for the Gaussian: `interp1d` localises each position on `linspace(0, 1, T)`, so its own float64 error
grows with T, and a bit-equality test against it fails at long T through scipy's error.  The oracle here therefore:

  Gaussian     scipy.ndimage.gaussian_filter1d(mode='reflect') on the input dtype: exact by definition;
  spline       the not-a-knot solve of the smoothed samples in np.longdouble, unit spacing (6 M1 = rhs1, 6 M(T-2) = rhs(T-2),
               Thomas on rows 2..T-3, M0 and M(T-1) extrapolated);
  evaluation   at s_i = i (T-1) / (kT-1) in long double, in interval min(floor(s_i), T-2), with the bound
               delta_i = 8 eps64 sum_q |a_q| + |p'(tt)| ulp64(s_i) of the float64 Horner step and position rounding.

Criteria (each test prints its worst error over the tolerance):

  Gaussian     a0 of the workspace equals the float32 scipy-smoothed sample, bit for bit;
  spline       a1, a2, a3 of the workspace within 64 eps64 max|y_col| of the long-double solve;
  evaluation   every output is the float32 rounding of some value in [truth - delta, truth + delta] (the positions where
               that interval straddles a rounding boundary are counted and printed).  Agreement with scipy's float32 cast
               is printed, not asserted: on inputs that cross zero, the correctly rounded truth itself differs from it at
               a few positions in a million already at T = 100;
  backward     per entry |gx - ref| <= ulp32(ref) / 2 + 1e-12 max|ref_col| against the float64 adjoint of
               tests/test_upsampling_backward_gpu.py;
  fused        the fused launches equal the two-launch path (pad_frames, then the radar launch) bit for bit; the synthesis
               adjoint from the cubics equals the one on the materialised batch within the stage-level tolerances of
               tests/test_backward_property_gpu.py.

The CPU tests pin the oracle to scipy (short sequences) and to CubicSpline's coefficients, show that the criteria reject
four deliberately wrong variants, and check that the fixed case table reaches every launch regime of the host plan
(vr_plan_pad_frames)."""
import ctypes

import numpy as np
import pytest
import torch
from hypothesis import HealthCheck, given, settings, strategies as st
from scipy.interpolate import CubicSpline
from scipy.ndimage import gaussian_filter1d

from oracle import backward as ob
from oracle import pad_frames as opf
from tests.test_upsampling_backward_gpu import pad_frames_adjoint

LD = np.longdouble
EPS64 = 2.0 ** -52
SMS = 148
needs_ld = pytest.mark.skipif(np.finfo(LD).nmant < 63, reason="np.longdouble has a %d-bit mantissa here; the oracle needs "
                              "x87 extended precision (63 bits)" % np.finfo(LD).nmant)

# ---- the case table -------------------------------------------------------------------------------------------------
# the dataset variant (vr_pad_frames_f32 / its backward / the spline-only launch): (N, T, V, M, k, sigma)
DATASET_CASES = [
    (1, 10240, 2, 1, 7, 3),        # the longest T: one column per CTA, forward and backward
    (1, 1000, 25, 2, 3, 3),        # ragged column blocks 13/13/13/11; 1024 % 13 != 0
    (256, 16, 3, 1, 2, 1),         # more units than 4 CTAs per SM: the grid-stride loop
    (2, 100, 25, 2, 5, 2),         # backward: 50 columns in one block, two 32-column groups
    (2, 4, 5, 1, 250, 10),         # T = 4 with the largest radius, 40 >= 2T: the reflection folds several times
    (1, 5, 3, 2, 8, 2.5),          # T = 5
    (1, 6, 4, 2, 250, 10),         # radius >= 2T with long k
    (3, 35, 7, 3, 1, 1.5),         # k = 1; T just above the clamp of the backward's Thomas coefficients
    (1, 300, 5, 1, 250, 3),        # the reference's T and k
]
# the notebook variant (vr_pad_frames_joints): (N, T, V, C, k, sigma, float64 input)
NOTEBOOK_CASES = [
    (1, 300, 5, 3, 250, 3, False),  # 18 row slices, 75000 % 18 != 0; V = 5 < 2r + 1 = 25
    (2, 8533, 2, 1, 2, 1, True),    # the longest T; C = 1
    (1, 64, 4, 2, 40, 10, True),    # C = 2, V far below the radius
    (3, 40, 6, 4, 9, 2, False),     # C = 4
]


# ---- the oracle ---------------------------------------------------------------------------------------------------------
def smooth(x, sigma, axis):
    """scipy's Gaussian (reflect boundary, result in the input dtype): the reference, exact by definition."""
    return gaussian_filter1d(x, float(sigma), axis=axis, mode="reflect")


def spline_coefficients(y, natural=False):
    """y (T, C) -> (T-1, 4, C) long double: the cubic a0 + a1 tt + a2 tt^2 + a3 tt^3 of every interval, unit spacing, of
    the not-a-knot spline through y (natural=True: the natural spline, a deliberately wrong variant)."""
    y = np.asarray(y).astype(LD)
    T = y.shape[0]
    rhs = 6 * ((y[:-2] - 2 * y[1:-1]) + y[2:])                 # rhs_i at index i - 1, i = 1 .. T-2
    M = np.zeros_like(y)
    if natural:                                                # M0 = M(T-1) = 0, rows 1 .. T-2
        lo, hi, d = 1, T - 2, rhs.copy()
    else:                                                      # 6 M1 = rhs1, 6 M(T-2) = rhs(T-2), rows 2 .. T-3
        M[1], M[T - 2] = rhs[0] / 6, rhs[T - 3] / 6
        lo, hi, d = 2, T - 3, rhs.copy()
        if lo <= hi:
            d[lo - 1] -= M[1]
            d[hi - 1] -= M[T - 2]
    if lo <= hi:                                               # Thomas: diagonal 4, off-diagonals 1
        cp = np.zeros(T, dtype=LD)
        dp = np.zeros_like(y)
        c, prev = LD(0), np.zeros_like(y[0])
        for i in range(lo, hi + 1):
            c = 1 / (4 - c)
            cp[i] = c
            prev = (d[i - 1] - prev) * c
            dp[i] = prev
        M[hi] = dp[hi]
        for i in range(hi - 1, lo - 1, -1):
            M[i] = dp[i] - cp[i] * M[i + 1]
    if not natural:
        M[0] = 2 * M[1] - M[2]
        M[T - 1] = 2 * M[T - 2] - M[T - 3]
    return np.stack([y[:-1], (y[1:] - y[:-1]) - (2 * M[:-1] + M[1:]) / 6, M[:-1] / 2, (M[1:] - M[:-1]) / 6], 1)


def evaluate(coef, T, k, last_in_last_interval=False, horner32=False, scipy_positions=False):
    """The spline at the k*T output positions -> (truth (kT, C) long double, delta (kT, C) float64).

    scipy_positions: delta also covers scipy's own float64 positions, which live on linspace(0, 1, .) rather than in unit
    spacing: each output position and the knot next to it is rounded there, i.e. up to 2 (T-1) ulp64(s_i / (T-1)) in s.

    last_in_last_interval / horner32: deliberately wrong variants -- the last position located in interval T-1 (tt = 0)
    while the cubic read is the last one there is; Horner's rule in float32."""
    KT = k * T
    s = np.arange(KT).astype(LD) * LD(T - 1) / LD(KT - 1)
    j = np.minimum(np.floor(s).astype(np.int64), T - 2)
    tt = s - j
    if last_in_last_interval:
        tt[-1] = s[-1] - np.floor(s[-1])
    a = coef[j]                                                # (KT, 4, C)
    t = tt[:, None]
    if horner32:
        a32, t32 = a.astype(np.float32), t.astype(np.float32)
        v = (a32[:, 0] + t32 * (a32[:, 1] + t32 * (a32[:, 2] + t32 * a32[:, 3]))).astype(LD)
    else:
        v = a[:, 0] + t * (a[:, 1] + t * (a[:, 2] + t * a[:, 3]))
    dp = a[:, 1] + t * (2 * a[:, 2] + 3 * t * a[:, 3])
    ds = np.spacing(s.astype(np.float64))
    if scipy_positions:
        ds = ds + 2 * (T - 1) * np.spacing((s / (T - 1)).astype(np.float64))
    delta = 8 * EPS64 * np.abs(a).sum(1).astype(np.float64) + np.abs(dp).astype(np.float64) * ds[:, None]
    return v, delta


def oracle_columns(y, k, natural=False, **variant):
    """Smoothed samples y (T, C) -> (coefficients, truth, delta)."""
    coef = spline_coefficients(y, natural)
    v, delta = evaluate(coef, y.shape[0], k, **variant)
    return coef, v, delta


def adjoint_with_scale(g, T, k, sigma):
    """The float64 adjoint of pad_frames and each entry's column scale max|ref| over time (axis -3)."""
    ref = pad_frames_adjoint(g, T, k, sigma)
    return ref, np.broadcast_to(np.abs(ref).max(axis=-3, keepdims=True), ref.shape)


def _reflect_once(t, T):
    t = np.where(t < 0, -t - 1, t)
    return np.clip(np.where(t >= T, 2 * T - t - 1, t), 0, T - 1)


def smooth_single_reflection(x, sigma, axis):
    """A deliberately wrong Gaussian: one reflection at each end, then clamped, instead of scipy's periodic 2T fold."""
    r = int(4 * float(sigma) + 0.5)
    w = np.exp(-0.5 / float(sigma) ** 2 * np.arange(-r, r + 1) ** 2)
    w /= w.sum()
    X = np.moveaxis(np.asarray(x, np.float64), axis, 0)
    T = X.shape[0]
    t = np.arange(T)
    acc = sum(w[o + r] * X[_reflect_once(t + o, T)] for o in range(-r, r + 1))
    return np.moveaxis(acc.astype(np.asarray(x).dtype), 0, axis)


# ---- the criteria -------------------------------------------------------------------------------------------------------
def gaussian_check(a0, ys):
    """a0 of the kernel's cubics (T-1, C) against the smoothed samples: bit-equal -> number of differing entries."""
    return int(np.count_nonzero(np.asarray(a0, np.float64) != np.asarray(ys[:-1], np.float64)))


def spline_check(a, coef, y):
    """max over a1..a3 of |kernel - long double| / (64 eps64 max|y_col|)."""
    tol = 64 * EPS64 * np.abs(np.asarray(y, np.float64)).max(0)
    err = np.abs(np.asarray(a[:, 1:], np.float64) - coef[:, 1:].astype(np.float64))
    return _ratio(err, np.broadcast_to(tol, err.shape))


def evaluation_check(out, v, delta):
    """out (kT, C) float32 -> (positions that are not the float32 rounding of a value in [v - delta, v + delta],
    positions where that interval straddles a rounding boundary, worst |out - v| / (delta + ulp32 / 2))."""
    lo, hi = (v - delta).astype(np.float32), (v + delta).astype(np.float32)
    out = np.asarray(out, np.float32)
    bad = int(np.count_nonzero(~((out >= lo) & (out <= hi))))
    straddle = int(np.count_nonzero(lo != hi))
    half_ulp = 0.5 * np.spacing(np.abs(v).astype(np.float32) + np.float32(0)).astype(np.float64)
    err = np.abs((out.astype(LD) - v).astype(np.float64))
    return bad, straddle, _ratio(err, delta + half_ulp)


def backward_check(gx, ref, colmax):
    """per entry |gx - ref| over ulp32(ref) / 2 + 1e-12 max|ref_col|."""
    tol = 0.5 * np.spacing(np.abs(ref).astype(np.float32)).astype(np.float64) + 1e-12 * colmax
    return _ratio(np.abs(np.asarray(gx, np.float64) - ref), tol)


def _ratio(diff, tol):
    """max diff / tol; an entry with tol == 0 must have diff == 0 exactly (inf otherwise)."""
    diff, tol = np.asarray(diff, np.float64), np.asarray(tol, np.float64)
    if np.any((tol == 0) & (diff != 0)):
        return np.inf
    sel = tol > 0
    return float((diff[sel] / tol[sel]).max()) if sel.any() else 0.0


def _columns(a, axis):
    """Move `axis` (time) to the front and flatten the rest into columns."""
    a = np.moveaxis(np.asarray(a), axis, 0)
    return a.reshape(a.shape[0], -1)


def _inputs(shape, seed, dtype=np.float32):
    """Zero-mean inputs without a ramp, so that the spline crosses zero."""
    return (np.random.default_rng(int(seed)).standard_normal(shape) * 0.5).astype(dtype)


# ---- CPU: the oracle ----------------------------------------------------------------------------------------------------
@needs_ld
@pytest.mark.parametrize("T,k,sigma", [(4, 250, 10), (5, 1, 1), (6, 13, 2.5), (40, 8, 3), (123, 7, 1.5), (300, 25, 3)])
def test_oracle_equals_scipy_on_short_sequences(T, k, sigma):
    """The long-double oracle equals scipy's float64 Dataset.pad_frames and notebook pad_frames within delta, widened by
    scipy's own float64 errors: its positions live on linspace(0, 1, .), and its banded solve may be off by the spline
    criterion's 64 eps64 max|y_col| in each of a1..a3."""
    def err(ref, y):
        _, v, delta = oracle_columns(y, k, scipy_positions=True)
        delta = delta + 3 * 64 * EPS64 * np.abs(y).max(0)
        return _ratio(np.abs((ref.astype(LD) - v).astype(np.float64)), delta)
    x = _inputs((3, T, 4, 2), T * 10 + k)
    e = err(_columns(opf.dataset_pad_frames(x, k, sigma), 1), _columns(smooth(x, sigma, 1), 1))
    xn = _inputs((T, 5, 3), T + k, np.float64)
    e_nb = err(_columns(opf.pad_frames(xn, k, sigma), 0), _columns(smooth(xn, sigma, 1), 0))
    print("T=%d k=%d sigma=%g: |scipy - oracle| / delta %.2e (dataset), %.2e (notebook)" % (T, k, sigma, e, e_nb))
    assert e <= 1 and e_nb <= 1


@needs_ld
@pytest.mark.parametrize("T", [4, 5, 6, 35, 300, 3000, 10240])
def test_oracle_coefficients_equal_cubic_spline(T):
    y = _inputs((T, 3), T).astype(np.float64)
    coef = spline_coefficients(y)
    c = CubicSpline(np.arange(T), y, bc_type="not-a-knot").c          # (4, T-1, C), highest power first
    err = np.abs(coef.astype(np.float64) - np.moveaxis(c[::-1], 0, 1)).max() / np.abs(y).max()
    print("T=%d: |oracle - CubicSpline| / max|y| %.2e" % (T, err))
    assert err <= 1e-14


@needs_ld
def test_criteria_reject_wrong_variants():
    """Four deliberately wrong up-samplings, run through the criteria the GPU tests apply: each is rejected, while the
    correctly rounded oracle passes.  T = 6 with sigma = 10 puts the radius (40) beyond 2T."""
    cases = [(6, 250, 10), (40, 25, 3), (300, 7, 2)]
    rejected = {}
    for T, k, sigma in cases:
        x = _inputs((3, T, 3, 2), 7 * T + k)
        ys = _columns(smooth(x, sigma, 1), 1)
        coef, v, delta = oracle_columns(ys, k)
        assert gaussian_check(coef[:, 0], ys) == 0
        assert spline_check(coef.astype(np.float64), coef, ys) <= 1
        assert evaluation_check(v.astype(np.float32), v, delta)[0] == 0
        variants = {"natural end conditions": oracle_columns(ys, k, natural=True),
                    "last position in interval T-1": oracle_columns(ys, k, last_in_last_interval=True),
                    "Horner in float32": oracle_columns(ys, k, horner32=True)}
        if 4 * sigma + 0.5 >= T:
            yw = _columns(smooth_single_reflection(x, sigma, 1), 1)
            variants["single reflection"] = (spline_coefficients(yw),) + evaluate(spline_coefficients(yw), T, k)
        for name, (cw, vw, _) in variants.items():
            g = gaussian_check(cw[:, 0], ys)
            s = spline_check(cw.astype(np.float64), coef, ys)
            bad, _, e = evaluation_check(vw.astype(np.float32), v, delta)
            print("%-30s T=%d k=%d sigma=%g: a0 differing %d, spline %.2e, evaluation: %d positions outside, %.2e"
                  % (name, T, k, sigma, g, s, bad, e))
            assert bad > 0, (name, T, k, sigma)
            rejected[name] = True
            if name in ("natural end conditions",):
                assert s > 1
            if name == "single reflection":
                assert g > 0
    assert set(rejected) == {"natural end conditions", "last position in interval T-1", "Horner in float32",
                             "single reflection"}


# ---- CPU: the launch plans ----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def cabi():
    import __graft_entry__ as ge
    ge.build_product()
    from skeleton_action_recognition_b200 import _cabi
    return _cabi


def _regimes(cabi, sm_count):
    """Which launch regimes the case table reaches, by the host plan with `sm_count` SMs."""
    seen = set()
    for N, T, V, M, k, sigma in DATASET_CASES:
        f = cabi.plan_pad_frames("forward", N, T, V, M, k, sigma, sm_count)
        b = cabi.plan_pad_frames("backward", N, T, V, M, k, sigma, sm_count)
        VM = V * M
        last = VM - (f["ncb"] - 1) * f["nc"]
        assert 1 <= last <= f["nc"] and f["units"] == 3 * N * f["ncb"] and f["grid"] == min(f["units"], 4 * sm_count)
        assert f["smem_bytes"] <= 227 * 1024 and b["smem_bytes"] <= 227 * 1024 and f["radius"] == int(4 * sigma + 0.5)
        seen |= {"T<=5"} if T <= 5 else set()
        seen |= {"T>34"} if T > 34 else set()
        if f["nc"] == 1 and T == 10240:
            seen.add("forward nc=1")
        if f["ncb"] > 1 and last != f["nc"]:
            seen.add("ragged column blocks")
        if f["units"] > f["grid"]:
            seen.add("units > grid")
        if 1024 % f["nc"] or 1024 % last:
            seen.add("1024 % ncl != 0")
        if b["nc"] == 1:
            seen.add("backward nc=1")
        if (b["nc"] + 31) // 32 > 1:
            seen.add("backward ngr>1")
        if f["radius"] >= 2 * T:
            seen.add("radius >= 2T")
        if f["radius"] == 40:
            seen.add("radius 40")
    cs, dtypes = set(), set()
    for N, T, V, C, k, sigma, f64 in NOTEBOOK_CASES:
        p = cabi.plan_pad_frames("notebook", N, T, V, C, k, sigma, sm_count)
        assert p["units"] == N * p["ncb"] * p["nrs"] and p["nrs"] * p["rows_per_slice"] >= k * T
        assert (p["nrs"] - 1) * p["rows_per_slice"] < k * T and p["smem_bytes"] <= 227 * 1024
        if p["nrs"] > 1 and (k * T) % p["nrs"]:
            seen.add("notebook ragged row slices")
        if V < 2 * p["radius"] + 1:
            seen.add("notebook V < 2r+1")
        if T == 8533:
            seen.add("notebook T=8533")
        cs.add(C)
        dtypes.add(f64)
    if cs == {1, 2, 3, 4}:
        seen.add("C 1..4")
    if dtypes == {False, True}:
        seen.add("both dtypes")
    return seen


ALL_REGIMES = {"forward nc=1", "ragged column blocks", "units > grid", "1024 % ncl != 0", "backward nc=1", "backward ngr>1",
               "T<=5", "T>34", "radius >= 2T", "radius 40", "notebook ragged row slices", "notebook V < 2r+1",
               "notebook T=8533", "C 1..4", "both dtypes"}


def test_case_table_reaches_every_launch_regime(cabi):
    seen = _regimes(cabi, SMS)
    assert seen == ALL_REGIMES, ALL_REGIMES - seen
    p = cabi.plan_pad_frames("forward", 1, 1000, 25, 2, 3, 3)
    assert (p["nc"], p["ncb"]) == (13, 4)                         # 13/13/13/11
    assert cabi.plan_pad_frames("forward", 1, 10240, 2, 1, 7, 3)["nc"] == 1
    assert cabi.plan_pad_frames("backward", 1, 10240, 2, 1, 7, 3)["nc"] == 1
    assert cabi.plan_pad_frames("notebook", 1, 300, 5, 3, 250, 3)["nrs"] == 18


def test_plan_rejects_what_the_launches_reject(cabi):
    with pytest.raises(NotImplementedError, match="too long"):
        cabi.plan_pad_frames("forward", 1, 10241, 2, 1, 1, 3)
    with pytest.raises(NotImplementedError, match="too long"):
        cabi.plan_pad_frames("backward", 1, 10241, 2, 1, 1, 3)
    with pytest.raises(NotImplementedError, match="too long"):
        cabi.plan_pad_frames("notebook", 1, 8534, 2, 1, 1, 3)
    with pytest.raises(NotImplementedError, match="radius"):
        cabi.plan_pad_frames("forward", 1, 40, 2, 1, 1, 10.2)
    with pytest.raises(ValueError):
        cabi.plan_pad_frames("forward", 1, 3, 2, 1, 1, 3)
    with pytest.raises(ValueError):
        cabi.plan_pad_frames("notebook", 1, 40, 2, 0, 1, 3)
    assert cabi.lib().vr_plan_pad_frames(3, 1, 40, 2, 1, 1, ctypes.c_float(3.0), 148, (ctypes.c_int64 * 8)()) == cabi.VR_ERR_ARG


# ---- GPU ----------------------------------------------------------------------------------------------------------------
def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _edges(V):
    return [(i, i + 1) for i in range(min(V - 1, 16))] if V > 1 else [(0, 0)]


def _layer(V):
    from skeleton_action_recognition_b200 import VirtualRadar
    return VirtualRadar(edges=_edges(V), wavelength=1e-3, radar_location=[0.3, -0.2, 1.5], device="cuda:0").to("cuda:0")


def _workspace(layer, xc, k, sigma):
    """The spline-only launch's cubics as (T-1, 4, N*3*V*M) float64 columns, and the fused iq (N, kT, 2)."""
    iq, work = layer._synth_upsampled(xc, k, sigma)
    N, _, T, V, M = xc.shape
    w = work[: N * (T - 1) * 4 * 3 * V * M].view(N, T - 1, 4, 3 * V * M).permute(1, 2, 0, 3).reshape(T - 1, 4, -1)
    return w.cpu().numpy(), iq


def _bits(t):
    return t.contiguous().view(torch.int32)


def check_dataset(N, T, V, M, k, sigma, seed, fused=True):
    """The dataset variant's forward (Gaussian, spline, evaluation), backward and fused launches for one case."""
    from skeleton_action_recognition_b200 import _cabi, pad_frames
    tag = "N=%d T=%d V=%d M=%d k=%d sigma=%g" % (N, T, V, M, k, sigma)
    seed = int(seed)
    x = _inputs((N, 3, T, V, M), seed)
    xc = torch.from_numpy(x).cuda()
    layer = _layer(V)
    up = pad_frames(xc, k, sigma)
    a, iq = _workspace(layer, xc, k, sigma)
    ys = _columns(smooth(x, sigma, 2), 2)
    coef, v, delta = oracle_columns(ys, k)
    g_bad = gaussian_check(a[:, 0], ys)
    s_err = spline_check(a, coef, ys)
    bad, straddle, e_err = evaluation_check(_columns(up.cpu().numpy(), 2), v, delta)
    scipy_eq = np.nan
    if T * k * ys.shape[1] <= 2_000_000:
        ref = _columns(opf.dataset_pad_frames(x, k, sigma), 2).astype(np.float32)
        scipy_eq = float((ref == _columns(up.cpu().numpy(), 2)).mean())
    # backward: the kernel through the C ABI against the float64 adjoint
    g = _inputs((N, 3, k * T, V, M), seed + 1)
    gx = torch.empty_like(xc)
    _cabi.check(_cabi.lib().vr_pad_frames_backward_f32(torch.from_numpy(g).cuda().data_ptr(), N, T, V, M, k,
                                                       ctypes.c_float(float(sigma)), gx.data_ptr(), _stream()))
    ref_gx, colmax = adjoint_with_scale(g, T, k, sigma)
    b_err = backward_check(gx.cpu().numpy(), ref_gx, colmax)
    print("%s: a0 differing %d | spline %.2e | evaluation %d outside, %.2e, %d straddling | backward %.2e | "
          "agreement with scipy's float32 cast %.6f" % (tag, g_bad, s_err, bad, e_err, straddle, b_err, scipy_eq))
    assert g_bad == 0 and s_err <= 1 and bad == 0 and b_err <= 1, tag
    if fused:
        check_fused(layer, xc, up, iq, k, sigma, tag, seed)


def _synth_materialised(layer, up):
    """vr_synth_f32 on the up-sampled batch.  Its load ring holds three chunks for two teams, so it rejects the widest V*M
    the fused launch (one stage per team) takes; one team per CTA leaves room for them, with the same sums in the same
    order."""
    from skeleton_action_recognition_b200 import _cabi
    try:
        return layer._synth(up, 0)
    except NotImplementedError:
        _cabi.check(_cabi.lib().vr_set_tuning(4, 1, 0))
        try:
            return layer._synth(up, 0)
        finally:
            _cabi.check(_cabi.lib().vr_set_tuning(0, 0, 0))


def check_fused(layer, xc, up, iq, k, sigma, tag, seed):
    """Fused launches against the two-launch path: iq and spectrograms bit for bit, the synthesis adjoint within the
    stage-level tolerances."""
    from tests import test_backward_property_gpu as tbp
    N, _, T, V, M = xc.shape
    assert torch.equal(_bits(iq), _bits(_synth_materialised(layer, up))), tag
    KT = k * T
    if KT > 128:
        with torch.no_grad():
            assert torch.equal(_bits(layer.forward_upsampled(xc, k, sigma)), _bits(layer(up))), tag
            F = KT // 16 + 1
            for S in sorted({min(F + 3, 4096), max(1, F // 2), 64}):      # dense (S >= F) and sparse (S < F) images
                assert torch.equal(_bits(layer.forward_upsampled(xc, k, sigma, image_size=S)),
                                   _bits(layer.forward_image(up, S))), (tag, S)
    if V > 1 and N * KT * M * len(layer.src) <= 2_000_000:
        gen = torch.Generator().manual_seed(seed + 2)
        giq = torch.randn(N, KT, 2, generator=gen)
        edges = _edges(V)
        gp_ref, _ = tbp.synth_gpu(up, giq, edges, 1e-3, [0.3, -0.2, 1.5], 0, want_x=False)
        _, work = layer._synth_upsampled(xc, k, sigma)
        gp = torch.zeros(4, dtype=torch.float64, device="cuda")
        from skeleton_action_recognition_b200 import _cabi
        _cabi.check(_cabi.lib().vr_synth_adjoint_upsampled_f32(work.data_ptr(), giq.cuda().data_ptr(), N, T, V, M,
                                                               layer._src_c, layer._dst_c, len(layer.src),
                                                               layer.wavelength.data_ptr(), layer.radar_location.data_ptr(),
                                                               0, k, gp.data_ptr(), _stream()))
        ref = ob.synth_adjoint(up.cpu().numpy(), giq.numpy(), edges, 1e-3, [0.3, -0.2, 1.5], "seq")
        t_lam, t_loc, _ = tbp.tolerances(ref, edges)
        a, b = gp.cpu().numpy(), gp_ref.cpu().numpy()
        e_lam, e_loc = _ratio(abs(a[0] - b[0]), t_lam), _ratio(np.abs(a[1:] - b[1:]), t_loc)
        print("%s: synthesis adjoint from the cubics vs the materialised batch: lam %.2e loc %.2e" % (tag, e_lam, e_loc))
        assert e_lam <= 1 and e_loc <= 1, (tag, a, b)


def check_notebook(N, T, V, C, k, sigma, f64, seed):
    from skeleton_action_recognition_b200.upsample import pad_frames_notebook
    tag = "notebook N=%d T=%d V=%d C=%d k=%d sigma=%g %s" % (N, T, V, C, k, sigma, "float64" if f64 else "float32")
    x = _inputs((N, T, V, C), seed, np.float64 if f64 else np.float32)
    xd = torch.from_numpy(x).cuda()
    rows = pad_frames_notebook(xd, k, sigma)[..., 0].permute(0, 2, 3, 1)          # (N, kT, V, C)
    planar = pad_frames_notebook(xd, k, sigma, planar=True)[..., 0]             # (N, C, kT, V)
    assert torch.equal(planar.permute(0, 2, 3, 1), rows), tag
    ys = _columns(smooth(x, sigma, 2), 1)
    _, v, delta = oracle_columns(ys, k)
    bad, straddle, e_err = evaluation_check(_columns(rows.cpu().numpy(), 1), v, delta)
    print("%s: evaluation %d outside, %.2e, %d straddling" % (tag, bad, e_err, straddle))
    assert bad == 0, tag


@needs_ld
@pytest.mark.gpu
@pytest.mark.parametrize("case", DATASET_CASES, ids=lambda c: "N%d-T%d-V%d-M%d-k%d-s%g" % c)
def test_dataset_variant_regimes(case):
    check_dataset(*case, seed=sum(case) * 7 + 1)


@needs_ld
@pytest.mark.gpu
@pytest.mark.parametrize("case", NOTEBOOK_CASES, ids=lambda c: "N%d-T%d-V%d-C%d-k%d-s%g-%s" % (c[:6] + ("f64" if c[6] else "f32",)))
def test_notebook_variant_regimes(case):
    check_notebook(*case, seed=sum(case[:6]) * 3 + 1)


@needs_ld
@pytest.mark.gpu
@settings(max_examples=30, derandomize=True, deadline=None, suppress_health_check=list(HealthCheck))
@given(st.data())
def test_dataset_variant_random_draws(data):
    T = data.draw(st.one_of(st.integers(4, 40), st.integers(41, 1500), st.integers(1500, 10240)), label="T")
    k = data.draw(st.sampled_from([1, 2, 3, 7, 8, 25, 250]), label="k")
    if T * k > 120_000:
        k = max(1, 120_000 // T)
    sigma = data.draw(st.sampled_from([0.5, 1, 1.5, 2.5, 3, 5, 7.25, 10]), label="sigma")
    cols = max(1, 1_500_000 // (3 * T * k))                   # columns the CPU oracle can afford
    M = data.draw(st.integers(1, min(3, cols)), label="M")
    V = data.draw(st.integers(1, max(1, min(30, cols // M))), label="V")
    N = data.draw(st.integers(1, max(1, min(3, cols // (V * M)))), label="N")
    check_dataset(N, T, V, M, k, sigma, seed=T * 31 + k * 7 + V * 3 + M + N)


@needs_ld
@pytest.mark.gpu
@settings(max_examples=8, derandomize=True, deadline=None, suppress_health_check=list(HealthCheck))
@given(st.data())
def test_notebook_variant_random_draws(data):
    T = data.draw(st.one_of(st.integers(4, 60), st.integers(61, 8533)), label="T")
    k = data.draw(st.sampled_from([1, 2, 3, 7, 8, 25, 250]), label="k")
    if T * k > 100_000:
        k = max(1, 100_000 // T)
    sigma = data.draw(st.sampled_from([0.5, 1, 2.5, 3, 10]), label="sigma")
    C = data.draw(st.integers(1, 4), label="C")
    V = data.draw(st.integers(1, max(1, min(25, 1_000_000 // (T * k * C)))), label="V")
    check_notebook(1, T, V, C, k, sigma, data.draw(st.booleans(), label="f64"), seed=T + k + V + C)


@pytest.mark.gpu
def test_device_plan_reaches_the_grid_stride_loop(cabi):
    """With the device's own SM count, the case table still has more units than the grid."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert "units > grid" in _regimes(cabi, sms), sms


def _largest_fused_vm(M, T, k):
    """The largest V*M (V = VM / M) the fused up-sampled launch accepts for T raw frames up-sampled k times (the plan's z
    buffer, and with it the room left for stages, depends on the length), by bisection on VR_ERR_UNSUPPORTED.  Every probe
    gets a real workspace (the spline launch runs before the radar launch's plan is checked); a rejected probe must leave
    iq untouched."""
    from skeleton_action_recognition_b200 import _cabi
    L = _cabi.lib()
    lam = torch.tensor(1e-3, device="cuda")
    loc = torch.zeros(3, device="cuda")

    def accepted(V):
        x = torch.zeros(1, 3, T, V, M, device="cuda")
        nbytes = int(L.vr_upsampled_workspace_bytes(1, T, V, M))
        work = torch.empty(nbytes // 8, dtype=torch.float64, device="cuda")
        iq = torch.full((1, k * T, 2), 7.0, device="cuda")
        src, dst = _cabi.i32_array([0]), _cabi.i32_array([1 % V])
        rc = L.vr_synth_upsampled_f32(x.data_ptr(), 1, T, V, M, src, dst, 1, lam.data_ptr(), loc.data_ptr(), 0, k,
                                      ctypes.c_float(1.0), work.data_ptr(), nbytes, iq.data_ptr(), _stream())
        if rc == _cabi.VR_ERR_UNSUPPORTED:
            torch.cuda.synchronize()
            assert bool((iq == 7.0).all()), V
            return False
        _cabi.check(rc)
        return True

    lo, hi = 1, 16384 // M
    assert accepted(lo) and not accepted(hi)
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if accepted(mid) else (lo, mid)
    return lo * M


@needs_ld
@pytest.mark.gpu
def test_fused_evaluation_across_vm():
    """The fused launch's evaluation from the cubics: the specialised V*M = 50 (even M), generic V*M from 1 to the largest
    the launch accepts (one lane then does several items per chunk), that largest plus one rejected; odd M, k < 8 (items
    cross raw intervals), sigma up to 10."""
    vm_max, vm3 = _largest_fused_vm(1, 9, 7), _largest_fused_vm(3, 8, 3)
    print("largest V*M of the fused up-sampled launch: %d (M = 1, T = 9, k = 7), %d (M = 3, T = 8, k = 3)" % (vm_max, vm3))
    assert vm_max > 50 and vm3 > 50
    cases = [(2, 40, 25, 2, 7, 3), (1, 60, 25, 2, 250, 10), (1, 30, 1, 1, 8, 1), (2, 33, 5, 1, 3, 2.5), (1, 20, 11, 3, 2, 1.5),
             (1, 12, 13, 1, 1, 10), (1, 9, vm_max, 1, 7, 3), (1, 8, vm3 // 3, 3, 3, 2)]
    for N, T, V, M, k, sigma in cases:
        check_dataset(N, T, V, M, k, sigma, seed=N + T + V + M + k)
    with pytest.raises(NotImplementedError):
        _layer(vm_max + 1)._synth_upsampled(torch.zeros(1, 3, 9, vm_max + 1, 1, device="cuda"), 7, 3)
