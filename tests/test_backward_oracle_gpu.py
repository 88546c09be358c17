"""The backward kernels (csrc/vr_backward.cuh) stage by stage against float64, in every launch regime of the host plan
(vr_plan_backward): the owner-form adjoint STFT, the scalar and per-sequence synthesis adjoints and the per-sequence fold.

The test owns every buffer through the C ABI: x and the up-sampling workspace sit at the start of NaN-filled allocations,
gz is prefilled with a sentinel NaN payload the kernels never store (their own NaN is 0x7fc00000), and grad_params, dL/dx
and gz are followed by guard regions that must come back untouched.

Stage 1 -- the adjoint STFT (vr_stft_adjoint_kernel) from the float32 iq and grad_out it read.  Per frame f, in float64:
X = FFT(h zp), G_k = g_k X_k / (|X_k| (|X_k| + 1e-6)) with g_k the grad_out row (k + 128) mod 256, y = h conj(FFT(conj G)),
overlap-added at the frame's positions through both reflect mirrors.  The kernel's arithmetic (-fmad=false, no fast-math:
sqrtf and / are IEEE; u = 2^-24), term by term:

    h_n = fmaf(-0.5, cospif(n / 128), 0.5)       absolute 2^-24 + u h_n (cospif 1 ulp, times 0.5, the FMA)
    X = bwd_fft256(pscale(zp, h))                 gamma_1 = 25 u times sum |h zp|: the Hann product 1, two dft8 levels 6
                                                  each (one add level, the sqrt(1/2) scale: add_mj, the rounded constant, the
                                                  product; two add levels of the dft4), two twiddle pcmul 5 each (product and
                                                  FMA 2 sqrt 2 u, the sincospif table 1 ulp on cos and sin: sqrt 2 u), the
                                                  final dft4 2.  With the table's 2^-24 sum |zp|:
                                                  delta = gamma_1 sum |h zp| + 2^-24 sum |zp|
    a = sqrtf(x x + y y)                          2 u relative (two products and a sum: 2 u on a^2, u on a; the square root u),
                                                  and where x x + y y is subnormal an absolute 2^-74 (a^2 errs by <= 3 2^-150):
                                                  delta' = delta + 2^-74.  Below |X| ~ 2^-75 both squares flush to 0, a = 0 and
                                                  the kernel defines G = 0.
    s = g / (a (a + 1e-6)); tr = (s x, -s y)      rho = 7 u relative on G (a twice at 2 u, the add, the product, the division,
                                                  the final product)
    G's sensitivity to X                          per bin as an interval: with r = |X64| and r_lo = max(r - delta', 0), every
                                                  |Y - X64| <= delta' gives |G(Y) - G(X64)| <= 2 |g| delta' / (r_lo (r_lo + 1e-6))
                                                  (|dG| <= |g| |dY| (1 / (r (r + e)) + 1 / (r + e)^2)), capped at
                                                  3 |g| / (r_lo + 1e-6): |G64| <= |g| / (r + e), and in the subnormal range
                                                  the kernel's a may be 1/sqrt 2 of |X|, so |G_kernel| <= 2 |g| / (r_lo + e).
                                                  dG = S + rho (|G64| + S), S that sensitivity.  G = 0 lies inside.
    Y = bwd_fft256(conj G)                        gamma_2 = 24 u (no Hann product) times sum (|G64| + dG), plus sum dG
    y_n = h_n Y_n                                 the product u, the table's error times |Y|:
                                                  b_n = h_n E2 + (2^-24 + 2 u h_n) (|Y64_n| + E2),  E2 = sum dG + gamma_2 sum |G|
    overlap-add, float32, in frame order          c_t u sum |y| for the c_t contributions to sample t

so |gz_gpu(t) - gz64(t)| <= SAFETY (sum of b over the contributions to t + c_t u sum |y|).  A sample no frame covers has
bound 0 and must be bitwise +0.0.  In the well-conditioned cases the test zeroes grad_out on every (bin, frame) whose
|X64| < 2^-5 sum |h zp|: the kernel then multiplies exact zeros there and the bound is tight (at 2^-8 the worst remaining
bins carry a 4e-4 relative bound and a dropped mirror misses by only 90x); the tiny-frame case scales iq by
2^-80, where float32 |X|^2 flushes to 0 and the kernel returns G = 0 (float64 gives |G| ~ 1e6 |g|): the interval admits it.

Stage 2 -- the synthesis adjoints (vr_synth_adjoint_kernel, vr_synth_adjoint_ups_kernel, vr_synth_adjoint_ps_kernel<UPS,
VIEWS> and vr_param_fold_kernel) from the gz the GPU left in stage 1, or from a dL/d(iq) the test chooses through
vr_synth_adjoint_f32 / vr_synth_adjoint_upsampled_f32, against oracle/backward.py:synth_adjoint with the tolerances of
tests/test_backward_property_gpu.py: 1e-12 sum |term| per parameter (per output for the per-sequence routes) and
4 k u S per dL/dx entry, k its float32 additions (R k with views).  Up-sampled positions: the GPU's own pad_frames output,
bit-identical to what the fused evaluation computes (tests/test_upsampling_kernels_gpu.py).  The oracle runs in time
chunks: parameter sums add across chunks, dL/dx is per step.

SAFETY = 2 covers the second-order terms the lists drop.  Each case prints its worst err/bound per stage.

The CPU tests pin stage 1 to oracle.backward.stft_adjoint and to float64 torch autograd of vro.stft_logmag; run a float32
numpy emulation of the kernel with every approximate instruction pushed to its documented error through the checker
(accepted at err/bound <= 0.5); show that eleven wrong variants miss by >= 100x; and check through vr_plan_backward at 148
SMs that the case table reaches every regime."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import backward as ob
from oracle import virtual_radar_oracle as vro
from tests import test_backward_property_gpu as bp
from tests import test_fused_forward_oracle_gpu as fw

U = 2.0 ** -24
SAFETY = 2.0
SMS = 148
GAMMA_1, GAMMA_2 = 25 * U, 24 * U
RHO = 7 * U
SUBNORMAL_ABS = 2.0 ** -74
TAU = 2.0 ** -5
SENTINEL = 0x7FB0DEAD
GUARD = 64
NTU = vro.NTU_EDGES
PREFILL = np.array([1.5, -2.25, 3.0, 0.125])


def _chain(n):
    return [(i, i + 1) for i in range(n)]


# ---- the case table ------------------------------------------------------------------------------------------------------
# entry: "backward" vr_backward_f32 (stage 1 + 2) / "params" vr_backward_params_f32 / "synth" vr_synth_adjoint_f32 /
#   "ups" vr_backward_upsampled_params_f32 / "ups_synth" vr_synth_adjoint_upsampled_f32.  T raw; K up-sampling factor.
# opts: gx (dL/dx wanted), ps (VR_FLAG_PER_SEQUENCE), views=R, fma, tiny (iq x 2^-80), geometry ("at-radar": a source joint
#   at the radar, "pointing": bones pointing at the radar), absent (second body zero), check (outputs checked; default all)
SMALL = [(0, 1), (1, 2), (1, 3)]
CASES = [
    dict(id="one-seg", entry="backward", N=4, T=300, V=25, M=2, edges=NTU, hop=16, gx=True),
    dict(id="ragged-hop16", entry="params", N=2, T=2100, V=25, M=2, edges=NTU, hop=16, fma=True),
    dict(id="ragged-hop37", entry="backward", N=2, T=2100, V=25, M=1, edges=NTU, hop=37, gx=True, geometry="pointing"),
    dict(id="T129-hop1", entry="backward", N=3, T=129, V=25, M=2, edges=NTU, hop=1, gx=True, absent=True),
    dict(id="F1-hop200", entry="params", N=2, T=150, V=25, M=2, edges=NTU, hop=200),
    dict(id="last-round-short", entry="backward", N=2, T=300, V=4, M=1, edges=SMALL, hop=30, gx=True),
    dict(id="empty-segs-hop3000", entry="params", N=1, T=20000, V=4, M=1, edges=SMALL, hop=3000),
    dict(id="right-mirror-cut", entry="params", N=1, T=74880, V=4, M=1, edges=SMALL, hop=16),
    dict(id="tiny-frames", entry="params", N=2, T=300, V=25, M=2, edges=NTU, hop=16, tiny=True),
    dict(id="job-stride-N1200", entry="params", N=1200, T=300, V=4, M=1, edges=SMALL, hop=16, check=(0, 599, 1199)),
    dict(id="ps-N1200", entry="backward", N=1200, T=300, V=4, M=1, edges=SMALL, hop=16, ps=True, check=(0, 599, 1199)),
    dict(id="ps-gx-E128", entry="backward", N=3, T=300, V=129, M=1, edges=_chain(128), hop=16, ps=True, gx=True, fma=True),
    dict(id="ps-at-radar", entry="params", N=40, T=300, V=25, M=2, edges=NTU, hop=16, ps=True, geometry="at-radar"),
    dict(id="views2-rows", entry="backward", N=4, T=300, V=25, M=2, edges=NTU, hop=16, ps=True, views=2, gx=True),
    dict(id="views3-outputs", entry="params", N=6, T=300, V=25, M=2, edges=NTU, hop=16, ps=True, views=3),
    dict(id="views7-rows", entry="synth", N=7, T=100, V=25, M=1, edges=NTU, ps=True, views=7, gx=True),
    dict(id="views7-outputs", entry="synth", N=14, T=100, V=4, M=1, edges=SMALL, ps=True, views=7),
    dict(id="synth-T1", entry="synth", N=3, T=1, V=25, M=2, edges=NTU, gx=True),
    dict(id="synth-T7-ps", entry="synth", N=3, T=7, V=25, M=2, edges=NTU, ps=True, gx=True),
    dict(id="synth-wrap", entry="synth", N=1200, T=300, V=2, M=1, edges=[(0, 1)], gx=True),
    dict(id="ups-K250", entry="ups", N=32, T=300, V=4, M=1, edges=SMALL, hop=16, K=250, ps=True, check=(0, 31)),
    dict(id="ups-K240-cut", entry="ups", N=1, T=312, V=4, M=1, edges=SMALL, hop=16, K=240),
    dict(id="ups-scalar-K250", entry="ups_synth", N=2, T=300, V=4, M=1, edges=SMALL, K=250),
    dict(id="ups-views2", entry="ups_synth", N=4, T=40, V=25, M=2, edges=NTU, K=10, ps=True, views=2),
    dict(id="ups-ps-K3", entry="ups_synth", N=3, T=40, V=25, M=2, edges=NTU, K=3, ps=True, fma=True),
]
ENTRY = {"backward": "backward", "params": "backward_params", "synth": "synth_adjoint", "ups": "backward_upsampled_params",
         "ups_synth": "synth_adjoint_upsampled"}


def _flags(case):
    from skeleton_action_recognition_b200 import _cabi
    f = _cabi.VR_FLAG_RANGE_FMA if case.get("fma") else 0
    if case.get("ps"):
        f |= _cabi.VR_FLAG_PER_SEQUENCE
    if case.get("views"):
        f |= _cabi.views_flag(case["views"])
    return f


def _plan(case):
    from skeleton_action_recognition_b200 import _cabi
    src, dst = map(list, zip(*case["edges"]))
    return _cabi.plan_backward(ENTRY[case["entry"]], case["N"], case["T"], case["V"], case["M"], src, dst,
                               hop=case.get("hop", 16), flags=_flags(case), grad_x=bool(case.get("gx")),
                               num_pad_frames=case.get("K", 0), sm_count=SMS)


def _regimes(case):
    from skeleton_action_recognition_b200 import _cabi
    p = _plan(case)
    tags = set()
    N, hop = case["N"], case.get("hop", 16)
    T = case["T"] * case.get("K", 1)
    if p["stft"]:
        plan, segs = _cabi.plan_adjoint_stft(N, T, hop, SMS)
        tags.add("stft")
        if len(segs) == 1:
            tags.add("stft-one-segment")
        else:
            tags.add("stft-segments")
            if plan["segment_length"] >= 3968 and hop < 256:
                tags.add("stft-4k-halo")
            if any(T - 129 <= s0 <= T - 2 for s0, _, _, _ in segs[1:]):
                tags.add("stft-cut-in-right-mirror")
            if any(lo > hi for _, _, lo, hi in segs):
                tags.add("stft-empty-segment")
        if N * plan["segments"] > plan["grid"]:
            tags.add("stft-job-stride")
        F = T // hop + 1
        if F == 1:
            tags.add("F=1")
        if T == 129:
            tags.add("T=129")
        if hop == 1:
            tags.add("hop=1")
        if any(hi >= lo and (hi - lo + 1) % 8 for _, _, lo, hi in segs):
            tags.add("short-last-round")
        if max(((hi - lo) // 8 + 1) for _, _, lo, hi in segs if hi >= lo) >= 33:
            tags.add("33-rounds")
    k, vm = p["synth_kernel"], p["views_mode"]
    if k == "ps":
        tags.add("ps<%s,%s>" % ("true" if p["ups"] else "false", vm) + ("+gx" if p["grad_x_fill"] else ""))
        if p["units"] > 4 * p["grid"]:
            tags.add("ps-unit-stride")
        if 4 * N > 128:
            tags.add("fold>128")
        if p["ps_segments"] >= 2344:
            tags.add("fold-2344")
        if vm != "none":
            tags.add("views%d-%s" % (p["views"], vm))
    else:
        tags.add(k)
        if p["units"] > 128 * p["grid"]:
            tags.add(k + "-stride")
    if case["entry"] in ("synth", "ups_synth") and case["T"] % 32:
        tags.add("synth-T<32" if case["T"] < 32 else "synth-T%32")
    if case.get("K") == 250:
        tags.add("K=250")
    for o in ("fma", "tiny", "absent"):
        if case.get(o):
            tags.add(o)
    if case.get("geometry"):
        tags.add(case["geometry"])
    if len(case["edges"]) == 128:
        tags.add("E=128")
    return tags


REQUIRED = {
    "stft-one-segment", "stft-segments", "stft-4k-halo", "stft-cut-in-right-mirror", "stft-empty-segment", "stft-job-stride",
    "F=1", "T=129", "hop=1", "short-last-round", "33-rounds",
    "scalar", "scalar-stride", "scalar_ups", "ps<false,none>", "ps<false,none>+gx", "ps<false,outputs>", "ps<false,rows>+gx",
    "ps<true,none>", "ps<true,outputs>", "views2-rows", "views3-outputs", "views7-rows", "views7-outputs", "ps-unit-stride",
    "fold>128", "fold-2344", "synth-T<32", "synth-T%32", "K=250", "fma", "tiny", "absent", "at-radar", "pointing", "E=128",
}


# ---- inputs ---------------------------------------------------------------------------------------------------------------
def _inputs(case, seed=0):
    """x (N / R, 3, T, V, M) float32, wavelengths (N,) and locations (N, 3) per output"""
    N, T, V, M = case["N"], case["T"], case["V"], case["M"]
    R = case.get("views", 1)
    Nx = N // R
    g = torch.Generator().manual_seed(seed + 7 * T + V)
    pose = torch.randn(Nx, 3, 1, V, M, generator=g) * 0.3
    t = torch.arange(T, dtype=torch.float32)[None, None, :, None, None]
    x = pose + 0.05 * torch.sin(2 * np.pi * 3 * t / 300 + torch.rand(Nx, 3, 1, V, M, generator=g) * 6.3)
    x = x + 0.01 * torch.randn(Nx, 3, T, V, M, generator=g)
    loc = np.zeros((N, 3), np.float32)
    loc[1::2] = [0.3, -0.2, 1.5]
    lam = np.full(N, 1e-3, np.float32)
    if case.get("ps"):
        lam = (1e-3 * (1 + 0.25 * (np.arange(N) % 5))).astype(np.float32)
    if case.get("absent") and M > 1:
        x[:, :, :, :, 1] = 0
    if case.get("geometry") == "at-radar":               # joint 0 (the source of bones) exactly at the radar for 50 steps
        x[0, :, 100:150, 0, 0] = torch.from_numpy(loc[0])[:, None]
    if case.get("geometry") == "pointing":               # bones 0->1 pointing at the radar to ~1e-3 rad
        L = torch.from_numpy(loc[0])[None, :, None]
        d = x[:, :, :, 0, 0] - L
        d = d / d.norm(dim=1, keepdim=True)
        x[:, :, :, 1, 0] = x[:, :, :, 0, 0] + 0.03 * (d + 1e-3 * torch.randn(d.shape, generator=g))
    return x.contiguous(), lam, loc


def _grad_iq(N, T, seed):
    """a dL/d(iq) with some exactly-zero steps (the kernels skip them)"""
    g = np.random.default_rng(seed).normal(0, 1, (N, T, 2)).astype(np.float32)
    g[:, ::5] = 0
    return g


# ---- stage 1: the float64 oracle and its bound ----------------------------------------------------------------------------
def hann():
    n = np.arange(256)
    return 0.5 - 0.5 * np.cos(2 * np.pi * n / 256)


def _positions(T, hop, frames=None):
    F = T // hop + 1
    f = np.arange(F) if frames is None else np.asarray(frames)
    return f[:, None] * hop - 128 + np.arange(256)[None, :]


def _reflect(p, T):
    t = np.abs(p)
    return np.where(t >= T, 2 * (T - 1) - t, t)


def frames64(iq, gout, hop, roll=128):
    """per frame of one sequence: X (F, 256), G (F, 256), the kernel's gk (F, 256) and delta (F,).  iq (T, 2), gout (256, F)"""
    T = iq.shape[0]
    z = iq[:, 0].astype(np.float64) + 1j * iq[:, 1].astype(np.float64)
    zp = z[_reflect(_positions(T, hop), T)]
    h = hann()
    X = np.fft.fft(h * zp, axis=1)
    gk = np.asarray(gout, np.float64)[(np.arange(256) + roll) % 256].T      # bin k reads row (k + 128) mod 256
    a = np.abs(X)
    with np.errstate(divide="ignore", invalid="ignore"):
        G = np.where(a > 0, gk * X / (a * (a + 1e-6)), 0)
    delta = GAMMA_1 * np.abs(h * zp).sum(1) + U * np.abs(zp).sum(1)
    return X, G, gk, delta


def well_conditioned(iq, gout, hop):
    """grad_out with every (bin, frame) whose |X64| < tau sum |h zp| set to 0 (rows fftshifted, as the kernel reads them)"""
    T = iq.shape[0]
    z = iq[:, 0].astype(np.float64) + 1j * iq[:, 1].astype(np.float64)
    hz = hann() * z[_reflect(_positions(T, hop), T)]
    a = np.abs(np.fft.fft(hz, axis=1))
    small = a < TAU * np.abs(hz).sum(1, keepdims=True)                       # (F, k)
    g = np.array(gout, np.float32)
    g[np.roll(small.T, 128, axis=0)] = 0
    return g


def overlap(vals, T, hop, variant=None, segs=None):
    """overlap-add of per-frame values (F, 256) into (T,) through both mirrors.  variant: a wrong kernel"""
    F = vals.shape[0]
    p = _positions(T, hop)
    t = _reflect(p, T)
    keep = np.ones(p.shape, bool)
    if variant == "right mirror dropped":
        keep &= p < T
    out = np.bincount(t[keep].ravel(), weights=vals[keep].real.ravel(), minlength=T).astype(np.complex128)
    out += 1j * np.bincount(t[keep].ravel(), weights=vals[keep].imag.ravel(), minlength=T)
    if variant == "right mirror one too far":                   # right = t <= T - 1: the last sample's direct part again
        m = p == T - 1
        out[T - 1] += vals[m].sum()
    if variant in ("halo frame dropped", "frames start one late"):
        for k, (s0, s1, lo, hi) in enumerate(segs):
            if k == 0 and variant == "halo frame dropped":
                continue
            # the halo frame nearest the cut (the last one whose window starts in the previous segment), or the first frame
            drop = (s0 + 127) // hop if variant == "halo frame dropped" else lo
            m = (t >= s0) & (t < s1) & (np.arange(F)[:, None] == drop)
            out -= np.bincount(t[m], weights=vals[m].real, minlength=T) + 1j * np.bincount(t[m], weights=vals[m].imag, minlength=T)
    return out


def stage1_oracle(iq, gout, hop, variant=None, segs=None):
    """gz64 (T,) complex, bound (T,), contributions per sample (T,) of one sequence"""
    T = iq.shape[0]
    roll = 127 if variant == "fftshift off by one" else 128
    X, G, gk, delta = frames64(iq, gout, hop, roll)
    h = hann()
    if variant == "conj dropped":
        Y = np.fft.fft(G, axis=1)
    else:
        Y = np.fft.ifft(G, axis=1) * 256                                    # sum_k G_k e^{+j 2 pi k n / 256}
    y = Y if variant == "window applied once" else h * Y
    gz = overlap(y, T, hop, variant, segs)
    r = np.abs(X)
    dp = (delta + SUBNORMAL_ABS)[:, None]
    r_lo = np.maximum(r - dp, 0)
    ag = np.abs(gk)
    with np.errstate(divide="ignore", invalid="ignore"):
        sup = np.where(ag > 0, 2 * ag * dp / (r_lo * (r_lo + 1e-6)), 0)
    S = np.minimum(sup, 3 * ag / (r_lo + 1e-6))
    dG = S + RHO * (np.abs(G) + S)
    E2 = dG.sum(1, keepdims=True) + GAMMA_2 * (np.abs(G) + dG).sum(1, keepdims=True)
    b = h * E2 + (2.0 ** -24 + 2 * U * h) * (np.abs(Y) + E2)
    ones = np.ones_like(b)
    bsum = overlap(b + 0j, T, hop).real
    cnt = overlap(ones + 0j, T, hop).real
    ysum = overlap(np.abs(y) + 0j, T, hop).real
    bound = SAFETY * (bsum + cnt * U * ysum)
    return gz, bound, cnt


def stage1_check(gz, want, bound, cnt):
    """worst err/bound of gz (T, 2) float32; uncovered samples bitwise +0.0"""
    g = np.asarray(gz)
    unc = cnt == 0
    assert (g[unc].view(np.int32) == 0).all(), "an uncovered sample is not +0.0"
    err = np.abs(g[:, 0].astype(np.float64) + 1j * g[:, 1].astype(np.float64) - want)
    assert np.all(np.isfinite(err)), "non-finite dL/d(iq)"
    assert np.all(err[bound == 0] == 0)
    ok = bound > 0
    return float((err[ok] / bound[ok]).max()) if ok.any() else 0.0


# ---- stage 2 --------------------------------------------------------------------------------------------------------------
def synth_oracle(pos, giq, edges, lam, loc, mode, chunk=4096):
    """ob.synth_adjoint of one output over time chunks -> (lam, loc (3,), x, scales (lam, loc, x))"""
    T = pos.shape[1]
    g_lam, g_loc, s_lam, s_loc = 0.0, np.zeros(3), 0.0, np.zeros(3)
    gx, sx = np.zeros(pos.shape), np.zeros(pos.shape)
    for t0 in range(0, T, chunk):
        t1 = min(T, t0 + chunk)
        r = ob.synth_adjoint(pos[None, :, t0:t1], giq[None, t0:t1], edges, lam, loc, mode)
        g_lam += r["lam"]
        g_loc += r["loc"]
        gx[:, t0:t1] = r["x"][0]
        s_lam += bp._scale(r, "lam")
        s_loc += bp._scale(r, "loc")
        sx[:, t0:t1] = bp._scale(r, "x")[0]
    return g_lam, g_loc, gx, (s_lam, s_loc, sx)


def params_ratio(gp, lam, loc, s_lam, s_loc, prefill=PREFILL):
    """worst err/tolerance of the 4 gradients gp (added to `prefill`) against (lam, loc): 1e-12 sum |term|, plus the
    rounding of the float64 add onto the prefill"""
    gp = np.asarray(gp, np.float64)
    tol = 1e-12 * np.concatenate([[s_lam], s_loc]) + 2.0 ** -52 * np.abs(gp)
    return bp._ratio(gp - prefill - np.concatenate([[lam], loc]), tol)


def grad_x_ratio(gx, want, sx, k):
    """worst err/tolerance of dL/dx entries: 4 k u S, k float32 additions into joint v (R k with views)"""
    return bp._ratio(np.asarray(gx, np.float64) - want, 4 * k[:, None] * U * sx + 1e-12 * sx)


# ---- CPU: pins ------------------------------------------------------------------------------------------------------------
def _cpu_iq(T=300, seed=0, scale=1.0):
    g = np.random.default_rng(seed)
    t = np.arange(T)
    z = np.exp(1j * (0.3 * t + 0.002 * t * t)) * (1 + 0.3 * g.normal(size=T)) + 0.2 * (g.normal(size=T) + 1j * g.normal(size=T))
    return (np.stack([z.real, z.imag], 1) * scale).astype(np.float32)


def test_stage1_oracle_equals_the_backward_oracle_and_float64_autograd():
    """stage 1's gz64 is ob.stft_adjoint's and float64 torch autograd of vro.stft_logmag's, to 1e-12 of the peak"""
    for T, hop in ((300, 16), (129, 1), (150, 200), (2100, 37)):
        iq = _cpu_iq(T, seed=T)
        F = T // hop + 1
        go = np.random.default_rng(hop).normal(size=(256, F)).astype(np.float32)
        gz, _, _ = stage1_oracle(iq, go, hop)
        ref = ob.stft_adjoint(iq[None], go[None], hop=hop)[0]
        o = vro.OracleVirtualRadar(hop_length=hop, dtype=torch.float64)
        x = torch.from_numpy(iq.astype(np.float64))[None].requires_grad_(True)
        (vro.stft_logmag(x, o.stft, 256) * torch.from_numpy(go.astype(np.float64))[None]).sum().backward()
        ag = x.grad[0].numpy()
        peak = np.abs(ref).max()
        assert np.abs(gz.real - ref[:, 0]).max() <= 1e-12 * peak and np.abs(gz.imag - ref[:, 1]).max() <= 1e-12 * peak
        assert np.abs(gz.real - ag[:, 0]).max() <= 1e-10 * peak and np.abs(gz.imag - ag[:, 1]).max() <= 1e-10 * peak


# ---- CPU: a float32 emulation of the kernel -------------------------------------------------------------------------------
f32 = np.float32


def _fft256_f32(zr, zi, sign):
    """bwd_fft256 on (F, 256) float32 inputs in natural order -> bins (F, 256) as (re, im); twiddles pushed by 1 ulp"""
    lane = np.arange(32)

    def tw(e):
        a = np.pi * ((e % 256) * (2.0 / 256))
        return (np.cos(a) * (1 + sign * 2.0 ** -24)).astype(f32), (-np.sin(a) * (1 + sign * 2.0 ** -24)).astype(f32)
    v = [(zr[:, lane + 32 * q], zi[:, lane + 32 * q]) for q in range(8)]
    v = fw._dft8(v)
    for q in range(1, 8):
        v[q] = fw._pcmul(v[q], *tw(lane * q))
    X1r = np.stack([a[0] for a in v], 1).reshape(-1, 8, 8, 4)
    X1i = np.stack([a[1] for a in v], 1).reshape(-1, 8, 8, 4)
    v = fw._dft8([(X1r[:, :, a, :], X1i[:, :, a, :]) for a in range(8)])
    b4 = np.arange(4)
    for c in range(1, 8):
        v[c] = fw._pcmul(v[c], *tw(8 * b4 * c))
    X2r = np.stack([a[0] for a in v], 2)
    X2i = np.stack([a[1] for a in v], 2)
    outr = np.zeros(zr.shape, f32)
    outi = np.zeros(zr.shape, f32)
    for c in range(8):
        ys = fw._dft4(*[(X2r[:, :, c, b], X2i[:, :, c, b]) for b in range(4)])
        for d in range(4):
            kbin = np.arange(8) + 8 * c + 64 * d
            outr[:, kbin], outi[:, kbin] = ys[d]
    return outr, outi


def emulate_adjoint(iq, gout, hop, sign):
    """vr_stft_adjoint_kernel in float32 for one sequence; cospif and sincospif pushed by 1 ulp in the direction `sign`"""
    T = iq.shape[0]
    p = _positions(T, hop)
    t = _reflect(p, T)
    n = np.arange(256)
    h = fw._fma(f32(-0.5), (np.cos(np.pi * (n * (2.0 / 256))) * (1 - sign * 2.0 ** -23)).astype(f32), f32(0.5))
    zr = (iq[t, 0] * h).astype(f32)
    zi = (iq[t, 1] * h).astype(f32)
    xr, xi = _fft256_f32(zr, zi, sign)
    a = np.sqrt(((xr * xr).astype(f32) + (xi * xi).astype(f32)).astype(f32))
    g = np.asarray(gout, f32)[(n + 128) % 256].T
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        s = np.where(a > 0, g / ((a * (a + f32(1e-6)).astype(f32)).astype(f32)), f32(0)).astype(f32)
    yr, yi = _fft256_f32((s * xr).astype(f32), (-(s * xi)).astype(f32), sign)
    cr, ci = (h * yr).astype(f32), (-(h * yi)).astype(f32)
    acc = np.zeros((T, 2), f32)
    for f in range(p.shape[0]):                                     # frame order; direct, left mirror, right mirror
        for m in (p[f] >= 0) & (p[f] < T), p[f] < 0, p[f] >= T:
            np.add.at(acc, (t[f][m], 0), cr[f][m])
            np.add.at(acc, (t[f][m], 1), ci[f][m])
    return acc


@pytest.mark.parametrize("sign", [1.0, -1.0])
def test_bound_accepts_the_kernels_arithmetic(sign):
    """the emulation passes at err/bound <= 0.5 on well-conditioned and arbitrary grad_out, at several hops, and on tiny
    frames (|X|^2 flushed to 0, G = 0)"""
    worst = 0.0
    for T, hop, tiny, wc in ((300, 16, False, True), (300, 16, False, False), (129, 1, False, True), (700, 37, False, True),
                             (300, 16, True, False)):
        iq = _cpu_iq(T, seed=hop, scale=2.0 ** -80 if tiny else 1.0)
        go = np.random.default_rng(T).normal(size=(256, T // hop + 1)).astype(np.float32)
        if wc:
            go = well_conditioned(iq, go, hop)
        gz = emulate_adjoint(iq, go, hop, sign)
        want, bound, cnt = stage1_oracle(iq, go, hop)
        if tiny:
            X, _, _, _ = frames64(iq, go, hop)
            assert (np.abs(X) < 2.0 ** -75).any() and (np.abs(X) > 0).all()
        worst = max(worst, stage1_check(gz, want, bound, cnt))
    print("emulation err/bound %.3g" % worst)
    assert worst <= 0.5, worst


def _reject(fn):
    try:
        return fn()
    except AssertionError:
        return float("inf")


def test_bounds_reject_wrong_variants():
    """seven wrong adjoint STFTs and four wrong synthesis adjoints miss their bound by >= 100x"""
    from skeleton_action_recognition_b200 import _cabi
    import __graft_entry__ as ge
    ge.build_product()
    T, hop = 2100, 16
    iq = _cpu_iq(T, seed=3)
    go = well_conditioned(iq, np.random.default_rng(4).normal(size=(256, T // hop + 1)).astype(np.float32), hop)
    _, segs = _cabi.plan_adjoint_stft(2, T, hop, SMS)
    assert len(segs) > 1
    want, bound, cnt = stage1_oracle(iq, go, hop)

    def as_gz(z):
        return np.stack([z.real, z.imag], 1).astype(np.float32)
    assert stage1_check(as_gz(want), want, bound, cnt) <= 0.5
    for v in ("right mirror dropped", "right mirror one too far", "halo frame dropped", "frames start one late",
              "window applied once", "fftshift off by one", "conj dropped"):
        bad = as_gz(stage1_oracle(iq, go, hop, v, segs)[0])
        r = _reject(lambda: stage1_check(bad, want, bound, cnt))
        print("stage 1 variant %-26s rejected at %.3g x the bound" % (v, r))
        assert r >= 100, (v, r)
    # stage 2: one output's gradients from wrong inputs against the right ones
    x, lam, loc = _inputs(dict(N=4, T=70, V=25, M=2, views=2))
    x = x.numpy()
    g = _grad_iq(4, 70, 1)
    k = 2 * bp._counts(NTU, 25).astype(np.float64)

    def og(pos, gi):
        return synth_oracle(pos, gi, NTU, lam[1], loc[1], "seq")
    ref = og(x[0], g[1])                                                       # output 1 = view 1 of x sequence 0
    later = np.concatenate([x[0][:, 5:], x[0][:, -5:]], 1)                    # positions of the next interval (K = 5)
    drop = g[1].copy()
    drop[32:64] = 0                                                            # the second 32-step segment's partial
    tail = g[1].copy()
    tail[70 - 26:] += g[2][:26]                                                # 26 lanes t >= T reading the next output's steps
    variants = {"views read sequence n, not n / R": og(x[1], g[1]), "UPS interval off by one": og(later, g[1]),
                "PS segment partial dropped": og(x[0], drop), "tail lane contributes": og(x[0], tail)}
    for name, o in variants.items():
        gp = PREFILL + np.concatenate([[o[0]], o[1]])
        r = max(params_ratio(gp, ref[0], ref[1], ref[3][0], ref[3][1]), grad_x_ratio(o[2], ref[2], ref[3][2], k))
        print("stage 2 variant %-34s rejected at %.3g x the tolerance" % (name, r))
        assert r >= 100, (name, r)


def test_case_table_reaches_every_regime():
    """through vr_plan_backward at 148 SMs: every adjoint-STFT regime, every synthesis kernel and fold regime"""
    import __graft_entry__ as ge
    ge.build_product()
    got = set()
    for c in CASES:
        got |= _regimes(c)
    assert REQUIRED <= got, sorted(REQUIRED - got)


def test_plan_facts():
    """ps<true, ROWS> cannot be reached (the up-sampled entries take no dL/dx), the static-slot grid cap cannot bind at 148
    SMs, and the plan rejects what the entries reject"""
    from skeleton_action_recognition_b200 import _cabi
    import __graft_entry__ as ge
    ge.build_product()
    src, dst = map(list, zip(*NTU))
    f = _cabi.VR_FLAG_PER_SEQUENCE | _cabi.views_flag(2)
    for e in ("backward_upsampled_params", "synth_adjoint_upsampled", "backward_params"):
        with pytest.raises(ValueError):
            _cabi.plan_backward(e, 4, 300, 25, 2, src, dst, flags=f, grad_x=True, num_pad_frames=10)
    p = _cabi.plan_backward("synth_adjoint_upsampled", 4, 300, 25, 2, src, dst, flags=f, num_pad_frames=10)
    assert (p["synth_kernel"], p["ups"], p["views_mode"]) == ("ps", 1, "outputs")
    big = _cabi.plan_backward("backward", 100000, 75000, 25, 2, src, dst)
    assert big["grid"] == 16 * SMS < big["grid_cap"] == 2560
    for bad, exc in ((dict(N=0), ValueError), (dict(T=128), ValueError), (dict(n_fft=512), NotImplementedError),
                     (dict(flags=_cabi.VR_FLAG_NOISE), ValueError), (dict(flags=_cabi.views_flag(2)), ValueError),
                     (dict(N=3, flags=f), ValueError), (dict(hop=0), ValueError)):
        kw = dict(N=4, T=300, V=25, M=2, src=src, dst=dst, hop=16)
        kw.update(bad)
        with pytest.raises(exc):
            _cabi.plan_backward("backward", **kw)
    with pytest.raises(ValueError):
        _cabi.plan_backward("backward", 2, 300, 3, 1, [0], [3])
    with pytest.raises(ValueError):
        _cabi.plan_backward("backward_upsampled_params", 2, 3, 25, 2, src, dst, num_pad_frames=10)
    p = _cabi.plan_backward("backward", 6, 300, 25, 2, src, dst, flags=_cabi.VR_FLAG_PER_SEQUENCE | _cabi.views_flag(3),
                            grad_x=True)
    assert (p["views_mode"], p["grad_x_fill"]) == ("rows", 2 * 3 * 300 * 25 * 2)


# ---- GPU ------------------------------------------------------------------------------------------------------------------
def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _guarded(n, dtype=torch.float32, fill=None):
    """a tensor of n entries followed by GUARD sentinel entries -> (buffer, view of the first n)"""
    if dtype == torch.float64:
        buf = torch.full((n + GUARD,), SENTINEL | (SENTINEL << 32), dtype=torch.int64, device="cuda").view(torch.float64)
    else:
        buf = torch.full((n + GUARD,), SENTINEL, dtype=torch.int32, device="cuda").view(torch.float32)
    if fill is not None:
        buf[:n] = fill
    return buf, buf[:n]


def _guard_intact(buf, n):
    tail = buf[n:]
    want = SENTINEL | (SENTINEL << 32) if buf.dtype == torch.float64 else SENTINEL
    return bool((tail.view(torch.int64 if buf.dtype == torch.float64 else torch.int32) == want).all())


def _run(case):
    """the case's launches with owned buffers -> dict of host arrays"""
    from skeleton_action_recognition_b200 import _cabi, pad_frames
    L = _cabi.lib()
    N, T, V, M = case["N"], case["T"], case["V"], case["M"]
    R, K = case.get("views", 1), case.get("K", 0)
    Tu = T * K if K else T
    hop = case.get("hop", 16)
    src, dst = map(list, zip(*case["edges"]))
    sc, dc = _cabi.i32_array(src), _cabi.i32_array(dst)
    flags = _flags(case)
    ps = bool(flags & _cabi.VR_FLAG_PER_SEQUENCE)
    x, lam, loc = _inputs(case)
    lam_d = torch.from_numpy(lam if ps else lam[:1]).cuda()
    loc_d = torch.from_numpy((loc if ps else loc[:1]).reshape(-1)).cuda()
    xbuf = torch.full((x.numel() + 1024,), float("nan"), device="cuda")
    xbuf[:x.numel()] = x.reshape(-1).cuda()
    st = _stream()
    pa = (lam_d.data_ptr(), loc_d.data_ptr())
    res = {"x": x.numpy(), "lam": lam, "loc": loc}
    fwd = (xbuf.data_ptr(), N, T, V, M, sc, dc, len(src)) + pa
    iq = torch.empty(N, Tu, 2, device="cuda")
    if K:
        nbytes = int(L.vr_upsampled_workspace_bytes(N // R, T, V, M))
        work = torch.full((nbytes // 8 + 1024,), float("nan"), dtype=torch.float64, device="cuda")
        _cabi.check(L.vr_synth_upsampled_f32(*fwd, flags, K, ctypes.c_float(3.0), work.data_ptr(), nbytes, iq.data_ptr(), st))
        res["pos"] = pad_frames(x.cuda(), K, 3.0).cpu().numpy()
    elif case["entry"] != "synth":
        _cabi.check(L.vr_synth_f32(*fwd, flags, iq.data_ptr(), st))
    if case.get("tiny"):
        iq *= 2.0 ** -80
    ngp = _cabi.per_sequence_grad_doubles(N, Tu) if ps else 4
    npre = 4 * N if ps else 4
    gp_buf, gp = _guarded(ngp, torch.float64)
    gp[:npre] = torch.from_numpy(np.tile(PREFILL, npre // 4)).cuda()
    want_x = bool(case.get("gx"))
    nx = (N // R) * 3 * Tu * V * M
    gx_buf, gx = _guarded(nx) if want_x else (None, None)
    if case["entry"] in ("synth", "ups_synth"):
        giq = torch.from_numpy(_grad_iq(N, Tu, 11)).cuda()
        gz_buf, gz = _guarded(N * Tu * 2, fill=giq.reshape(-1))
        res["giq"] = giq.cpu().numpy()
        if K:
            _cabi.check(L.vr_synth_adjoint_upsampled_f32(work.data_ptr(), gz.data_ptr(), N, T, V, M, sc, dc, len(src), *pa, flags,
                                                         K, gp.data_ptr(), st))
        else:
            _cabi.check(L.vr_synth_adjoint_f32(xbuf.data_ptr(), gz.data_ptr(), N, T, V, M, sc, dc, len(src), *pa, flags,
                                               gp.data_ptr(), gx.data_ptr() if want_x else None, st))
    else:
        F = Tu // hop + 1
        go = np.random.default_rng(5).normal(size=(N, 256, F)).astype(np.float32)
        iq_h = iq.cpu().numpy()
        if not case.get("tiny"):
            for n in set(_checked(case)):
                go[n] = well_conditioned(iq_h[n], go[n], hop)
        go_d = torch.from_numpy(go).cuda()
        gz_buf, gz = _guarded(N * Tu * 2)
        if K:
            _cabi.check(L.vr_backward_upsampled_params_f32(work.data_ptr(), iq.data_ptr(), go_d.data_ptr(), N, T, V, M, sc, dc,
                                                           len(src), *pa, 256, hop, flags, K, gz.data_ptr(), gp.data_ptr(), st))
        else:
            _cabi.check(L.vr_backward_f32(xbuf.data_ptr(), iq.data_ptr(), go_d.data_ptr(), N, T, V, M, sc, dc, len(src), *pa,
                                          256, hop, flags, gz.data_ptr(), gp.data_ptr(), gx.data_ptr() if want_x else None, st))
        res["iq"], res["go"] = iq_h, go
    torch.cuda.synchronize()
    assert _guard_intact(gp_buf, ngp), "grad_params guard written"
    assert _guard_intact(gz_buf, N * Tu * 2), "gz guard written"
    assert int((gz.view(torch.int32) == SENTINEL).sum()) == 0, "gz sample left unwritten"
    res["gz"] = gz.view(N, Tu, 2).cpu().numpy()
    res["gp"] = gp[:npre].cpu().numpy().reshape(-1, 4)
    if want_x:
        assert _guard_intact(gx_buf, nx), "dL/dx guard written"
        res["gx"] = gx.view(N // R, 3, Tu, V, M).cpu().numpy()
    return res


def _checked(case):
    return case.get("check", range(case["N"]))


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c["id"] for c in CASES])
def test_backward_stage_by_stage(case):
    res = _run(case)
    N, R = case["N"], case.get("views", 1)
    hop = case.get("hop", 16)
    mode = "fma" if case.get("fma") else "seq"
    ps = bool(case.get("ps"))
    edges = case["edges"]
    V = case["V"]
    w1 = w2 = 0.0
    if "iq" in res:
        for n in _checked(case):
            want, bound, cnt = stage1_oracle(res["iq"][n], res["go"][n], hop)
            w1 = max(w1, stage1_check(res["gz"][n], want, bound, cnt))
    pos = res.get("pos", res["x"])
    giq = res["gz"] if "giq" not in res else res["giq"]
    k = R * bp._counts(edges, V).astype(np.float64)
    outs = list(_checked(case)) if ps else range(N)
    tot_lam, tot_loc, s_lam, s_loc = 0.0, np.zeros(3), 0.0, np.zeros(3)
    gx_want, gx_scale = {}, {}
    for n in outs:
        q = n if ps else 0                                                    # the scalar entries take one placement
        g_lam, g_loc, gx, sc = synth_oracle(pos[n // R], giq[n], edges, res["lam"][q], res["loc"][q], mode)
        if ps:
            w2 = max(w2, params_ratio(res["gp"][n], g_lam, g_loc, sc[0], sc[1]))
        else:
            tot_lam, tot_loc, s_lam, s_loc = tot_lam + g_lam, tot_loc + g_loc, s_lam + sc[0], s_loc + sc[1]
        if "gx" in res:
            gx_want[n // R] = gx_want.get(n // R, 0) + gx
            gx_scale[n // R] = gx_scale.get(n // R, 0) + sc[2]
    if not ps:
        w2 = max(w2, params_ratio(res["gp"][0], tot_lam, tot_loc, s_lam, s_loc))
    for xn, gw in gx_want.items():
        w2 = max(w2, grad_x_ratio(res["gx"][xn], gw, gx_scale[xn], k))
    if ps:
        assert np.isfinite(res["gp"]).all()
    print("%s: stage 1 err/bound %.3g, stage 2 err/tolerance %.3g" % (case["id"], w1, w2))
    assert w1 <= 1 and w2 <= 1, (case["id"], w1, w2)


@pytest.mark.gpu
def test_static_slots_wrap():
    """34 consecutive scalar launches, each checked: the ring of 32 static partial slots wraps and every launch still adds
    its gradient, with its counter re-armed"""
    from skeleton_action_recognition_b200 import _cabi
    L = _cabi.lib()
    case = dict(N=3, T=200, V=25, M=2)
    x, lam, loc = _inputs(case)
    g = _grad_iq(3, 200, 2)
    src, dst = map(list, zip(*NTU))
    want = [0.0, np.zeros(3), 0.0, np.zeros(3)]
    for n in range(3):
        o = synth_oracle(x[n].numpy(), g[n], NTU, lam[0], loc[0], "seq")
        want = [want[0] + o[0], want[1] + o[1], want[2] + o[3][0], want[3] + o[3][1]]
    xd, gd = x.cuda(), torch.from_numpy(g).cuda()
    lam_d, loc_d = torch.from_numpy(lam[:1]).cuda(), torch.from_numpy(loc[0]).cuda()
    first = None
    for i in range(34):
        buf, gp = _guarded(4, torch.float64, fill=torch.from_numpy(PREFILL).cuda())
        _cabi.check(L.vr_synth_adjoint_f32(xd.data_ptr(), gd.data_ptr(), 3, 200, 25, 2, _cabi.i32_array(src),
                                           _cabi.i32_array(dst), len(src), lam_d.data_ptr(), loc_d.data_ptr(), 0,
                                           gp.data_ptr(), None, _stream()))
        torch.cuda.synchronize()
        assert _guard_intact(buf, 4)
        got = gp.cpu().numpy()
        assert params_ratio(got, *want) <= 1, i
        first = got if first is None else first
        assert np.array_equal(got, first), i
