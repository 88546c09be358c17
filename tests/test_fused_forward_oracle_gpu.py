"""The fused forward kernel (csrc/vr_kernels.cuh: vr_fused_kernel and vr_team_kernel) stage by stage against float64, in
every launch regime of both schedules (the host plan: vr_plan_launch).

Each stage is compared with float64 computed from the float32 values that stage starts from, with a bound per entry built
from that entry's own terms.  The test owns every buffer, fills `iq` and `out` with a sentinel NaN payload the kernel never
writes (its own NaN is 0x7fc00000) and requires that no sentinel survives the launch: an unwritten sample or pixel fails.

Stage 1 -- the baseband z[n, t] from the float32 positions the launch read (x; for the _upsampled entries the output of
vr_pad_frames_f32, which the fused evaluation reproduces bit for bit).  The kernel reproduces bit for bit the float32
range phase theta of every source joint and the aspect cosine u and length l of every bone (oracle/range_phase.c:
range_phase_c, aspect_cosine_c, in the layout's rounding mode).  From those, in float64:

    c = (sum_b l_b / E)^2,   amp_b = sqrt(pi c) / ((1 - u_b^2) + c u_b^2),   z = sum_bodies sum_bones amp_b exp(j theta_src(b))

per output placement (per-sequence placements and views go in per output).  NaN exactly where some bone of some body has
fl32(u u) > 1.  The kernel's arithmetic, term by term (u = 2^-24, the unit roundoff):

    u2    = fl(u u)                                  relative u
    cbar  = fl(fl((s0 + s1) + (s2 + s3)) * fl(1/E))  s_h: one warp's sequential sum of its <= eg bone lengths (all >= 0):
                                                     relative eps_c = (eg + 4) u (eg - 1 adds, two fold levels, 1/E, product)
    cm1   = fma(cbar, cbar, -1)                      |d cm1| <= 2 c eps_c + u |c - 1|
    den   = fma(u2, cm1, 1)                          |d den| <= u^2 |d cm1| + |c - 1| u u^2 + u den  -> relative d den / den
    w     = rcp.approx.ftz(den)                      1 ulp <= 2^-23 relative (PTX ISA, rcp.approx.f32)
    W_j   = sum of w over the joint's n_j bones      (n_j - 1) u relative (positive terms)
    r     = th - kk (c1 + c2), Cody-Waite            first FMA exact (|r| < 8 and both terms on a 2^-21 grid); the second
                                                     rounds: u |r|; the constant: |kk| |2 pi - (c1 + c2)|
    __sincosf(r)                                     2^-21.41 absolute on [-pi, pi] for each of cos and sin (CUDA C++
                                                     Programming Guide, intrinsic functions table): sqrt(2) 2^-21.41 complex
    ar, ai = fma(W_j, cos_j, ar) ...                 one rounding per source joint of the group on a partial sum bounded by
                                                     the group's sum of |terms|: ns u
    zr    = fma(K, ar, zr), K = fl(fl(sqrt pi) cbar) eps_c + 2 u relative on K; one rounding per body: M u
    (z0 + z1) + (z2 + z3)                            2 u

so |z_gpu - z64| <= SAFETY sum_{bones, bodies} amp_b eps_b with, per bone,
eps_b = d den_b / den_b + 2^-23 + (n_j - 1) u + eps_c + 2 u + dphi + sqrt(2) 2^-21.41 + (ns + M + 2) u.  The first term is the
one that matters: den can be as small as c (~1e-3 for a bone pointing at the radar) while its absolute error stays ~3 u,
so that bone's weight is good to ~1e-4 only; a flat relative bound on sum |terms| would fail there.

Stage 2 -- the spectrogram from the I/Q the GPU left: reflect-pad by 128 (nnAudio center=True), the periodic Hann window
h_n = 0.5 - 0.5 cos(2 pi n / 256) in float64, a float64 FFT, ln(|X| + 1e-6) at row (k + 128) mod 256; for image launches
pixel (r, c) is the entry at row min(floor(r 256/S), 255) and frame col_frame(c), ATen's float32 index rule
(oracle/resize.py).  NaN exactly where the frame's window touches a NaN sample.  The error of X (stft_frame: radix
8 x 8 x 4) is bounded by delta = SAFETY (gamma_FFT sum_n |h_n z_n| + 2^-24 sum_n |z_n|), the second term the Hann table's
absolute error (cospif 1 ulp, times 0.5, then fmaf: <= 2^-24 + u h_n).  gamma_FFT counts the roundings on a path through
stft_frame, each bounded by u times the L1 norm of the inputs it combines, and every map on the path is a combination with
coefficients of modulus one:

    Hann multiply                                                              1
    dft8: one add level, the sqrt(1/2) scale (add_mj, the rounded constant
          R, the product), two add levels of the dft4                          6     (twice: 12)
    twiddle pcmul: the product and the FMA (2 sqrt 2 u) plus the sincospif
          table (1 ulp on cos and sin: sqrt 2 u)                               5     (twice: 10)
    dft4: two add levels                                                       2
    gamma_FFT = 25 u

The magnitude adds fmaf(x, x, y y) (2 u relative on |X|^2, u on |X|), sqrt.approx.ftz.f32 (2^-23 relative, PTX ISA) and
the add of 1e-6f: delta' = delta + SAFETY (|X| + delta)(u + 2^-23).  The check is an interval, so |X| ~ 0 needs no case:

    out in [ln(max(|X64| - delta', 0) + 1e-6 (1 - u)) - eps_log, ln(|X64| + delta' + 1e-6 (1 + u)) + eps_log]

with eps_log = SAFETY (u + max(2^-21.41, 3 2^-23 |ln v|)): the rounding of the add, and __logf's 2^-21.41 absolute on
[0.5, 2] or 3 ulp elsewhere (Programming Guide).  sqrt.approx.ftz flushes |X|^2 < 2^-126 to 0, inside the interval.

SAFETY = 2 covers the second-order terms the lists drop.  Each case prints err/bound of each stage (at most 1 passes; for
stage 2 the distance from ln(|X64| + 1e-6) to the output over the distance to the interval's end on that side).

The CPU tests pin stage 1 (float64 u, l, theta) to oracle.forward_hybrid's baseband and stage 2 to the float64 nnAudio
restatement; run a float32 numpy emulation of the kernel's order of operations, with every approximate instruction
replaced by the correctly rounded function plus a perturbation at its documented error, through both checkers (accepted
at err/bound <= 0.5); check that twelve wrong variants are rejected by a wide margin; and check through vr_plan_launch at
148 SMs that the case table reaches every regime of both schedules."""
import ctypes
import math

import numpy as np
import pytest
import torch

from oracle import resize
from oracle import virtual_radar_oracle as vro

U = 2.0 ** -24
SAFETY = 2.0
SMS = 148
SINCOS_ABS = 2.0 ** -21.41        # __sinf / __cosf on [-pi, pi], absolute
RCP_REL = 2.0 ** -23              # rcp.approx.ftz.f32, 1 ulp
SQRT_REL = 2.0 ** -23             # sqrt.approx.ftz.f32
LOG_ABS, LOG_ULP = 2.0 ** -21.41, 3.0     # __logf: absolute on [0.5, 2], ulp elsewhere
GAMMA_FFT = 25 * U
C1, C2 = np.float32(6.2831854820251465), np.float32(-1.7484556000744883e-7)
CW_ERR = abs(2 * math.pi - (float(C1) + float(C2))) + 2.0 ** -50      # |2 pi - (c1 + c2)|, with float64's own error
SENTINEL = 0x7FB0DEAD                                                   # a signalling-NaN payload the kernel never stores
NTU = vro.NTU_EDGES

# ---- the case table ------------------------------------------------------------------------------------------------------
# route: "debug" vr_forward_debug_f32 / "synth" vr_synth_f32 / "image" vr_forward_image_f32 (+ vr_synth_f32 for the I/Q) /
#   "ups_debug" vr_forward_upsampled_debug_f32 / "ups_synth" vr_synth_upsampled_f32 / "ups_image" vr_forward_upsampled_f32
#   with image_size (+ vr_synth_upsampled_f32) / "team" vr_set_schedule(1) + vr_forward_f32, stage 2 from the I/Q of a
#   cooperative debug launch on the same inputs / "ready": two back-to-back debug launches with VR_FLAG_INPUTS_READY.
# opts: fma (coordinate-innermost rounding), off (x 4 bytes off its 16-byte alignment), absent (second body zero),
#   late (second body absent from step L on), radial (bones at the radar: NaN samples), offaxis, ps (per-sequence
#   placements mixing origin and off-axis), views=R, noise, S (image size), K (up-sampling factor)


def _star(n):
    return [(0, i) for i in range(1, n + 1)]


def _chain(n):
    return [(i, i + 1) for i in range(n)]


MIXED = [(0, 1), (0, 2), (0, 3), (1, 4), (4, 5), (5, 6), (2, 7), (7, 8), (3, 9), (0, 1)]     # multi-bone joints, a duplicate
CASES = [
    dict(id="ntu-bulk", route="debug", N=4, T=300, V=25, M=2, edges=NTU, hop=16, late=170),
    dict(id="ntu-fma-offaxis", route="debug", N=3, T=300, V=25, M=2, edges=NTU, hop=16, fma=True, offaxis=True, absent=True),
    dict(id="nb1-T129", route="debug", N=3, T=129, V=25, M=1, edges=NTU, hop=8, offaxis=True),
    dict(id="nb2-generic-T320", route="debug", N=2, T=320, V=11, M=2, edges=MIXED, hop=37, fma=True),
    dict(id="F26-rows17-T319", route="debug", N=2, T=319, V=25, M=2, edges=NTU, hop=8),
    dict(id="park-one-job", route="debug", N=1, T=1800, V=25, M=2, edges=NTU, hop=16, offaxis=True),
    dict(id="jobs-park", route="debug", N=2, T=5000, V=25, M=2, edges=NTU, hop=16, late=4001),
    dict(id="jobs-zcap", route="debug", N=1, T=4000, V=129, M=1, edges=_chain(128), hop=16),
    dict(id="E128-one-cta", route="debug", N=2, T=300, V=129, M=1, edges=_chain(128), hop=16, fma=True),
    dict(id="noTMA-T301", route="debug", N=2, T=301, V=25, M=1, edges=NTU, hop=16),
    dict(id="x-offset", route="debug", N=2, T=300, V=25, M=2, edges=NTU, hop=16, off=True, fma=True),
    dict(id="tickets", route="debug", N=400, T=300, V=25, M=2, edges=NTU, hop=16),
    dict(id="E1", route="debug", N=3, T=300, V=2, M=3, edges=[(0, 1)], hop=100, offaxis=True),
    dict(id="star32", route="debug", N=2, T=300, V=33, M=2, edges=_star(32), hop=16),
    dict(id="hop200-tail", route="debug", N=2, T=399, V=25, M=2, edges=NTU, hop=200),
    dict(id="hop300-gaps", route="debug", N=1, T=5000, V=25, M=2, edges=NTU, hop=300, offaxis=True),
    dict(id="radial-nan", route="debug", N=2, T=800, V=6, M=2, edges=_chain(5), hop=16, radial=True, fma=True),
    dict(id="ps-mixed", route="debug", N=4, T=300, V=25, M=2, edges=NTU, hop=16, ps=True),
    dict(id="views3", route="debug", N=6, T=300, V=25, M=2, edges=NTU, hop=16, ps=True, views=3),
    dict(id="noise", route="debug", N=3, T=300, V=25, M=2, edges=NTU, hop=16, ps=True, noise=True),
    dict(id="ready", route="ready", N=3, T=300, V=25, M=2, edges=NTU, hop=16),
    dict(id="synth", route="synth", N=2, T=1000, V=25, M=2, edges=NTU, hop=16, offaxis=True),
    dict(id="ups-synth-K3", route="ups_synth", N=2, T=40, V=25, M=2, edges=NTU, hop=16, K=3),
    dict(id="ups-synth-K10", route="ups_synth", N=2, T=60, V=25, M=1, edges=NTU, hop=16, K=10, offaxis=True),
    dict(id="ups-debug-tail", route="ups_debug", N=2, T=133, V=25, M=2, edges=NTU, hop=200, K=3),
    dict(id="ups-debug", route="ups_debug", N=2, T=100, V=25, M=2, edges=NTU, hop=16, K=10, offaxis=True),
    dict(id="image-256-dense", route="image", N=2, T=300, V=25, M=2, edges=NTU, hop=16, S=256),
    dict(id="image-37-dense-scalar", route="image", N=2, T=300, V=25, M=2, edges=NTU, hop=16, S=37),
    dict(id="image-100-sparse", route="image", N=2, T=3000, V=25, M=2, edges=NTU, hop=16, S=100),
    dict(id="image-77-sparse-scalar", route="image", N=2, T=2500, V=25, M=2, edges=NTU, hop=32, S=77, offaxis=True),
    dict(id="ups-image-64", route="ups_image", N=2, T=100, V=25, M=2, edges=NTU, hop=16, K=3, S=64),
    dict(id="team-ntu", route="team", N=6, T=300, V=25, M=2, edges=NTU, hop=16, offaxis=True),
    dict(id="team-nb1", route="team", N=5, T=300, V=25, M=1, edges=NTU, hop=16),
    dict(id="team-nb2-fma", route="team", N=4, T=300, V=20, M=2, edges=_chain(19), hop=16, fma=True),
    dict(id="team-tickets", route="team", N=700, T=300, V=25, M=2, edges=NTU, hop=16, late=100),
]


def _flags(case):
    from skeleton_action_recognition_b200 import _cabi
    f = _cabi.VR_FLAG_RANGE_FMA if case.get("fma") else 0
    if case.get("ps") or case.get("views") or case.get("noise"):
        f |= _cabi.VR_FLAG_PER_SEQUENCE
    if case.get("views"):
        f |= _cabi.views_flag(case["views"])
    if case.get("noise"):
        f |= _cabi.VR_FLAG_NOISE
    if case["route"] == "ready":
        f |= _cabi.VR_FLAG_INPUTS_READY
    return f


def _plans(case):
    """vr_plan_launch of every launch the case makes"""
    from skeleton_action_recognition_b200 import _cabi
    src, dst = map(list, zip(*case["edges"]))
    r, K, S = case["route"], case.get("K", 0), case.get("S", 0)
    T = case["T"]
    flags = _flags(case) & ~_cabi.VR_FLAG_NOISE
    args = (case["N"], T, case["V"], case["M"], src, dst)
    kw = dict(hop=case["hop"], flags=flags, x_aligned=not case.get("off"), sm_count=SMS)
    if r in ("debug", "ready"):
        return [_cabi.plan_launch("debug", *args, **kw)]
    if r == "synth":
        return [_cabi.plan_launch("synth", *args, **kw)]
    if r == "image":
        return [_cabi.plan_launch("spectrogram", *args, image_size=S, **kw), _cabi.plan_launch("synth", *args, **kw)]
    if r == "ups_debug":
        return [_cabi.plan_launch("debug", *args, num_pad_frames=K, **kw)]
    if r == "ups_synth":
        return [_cabi.plan_launch("synth", *args, num_pad_frames=K, **kw)]
    if r == "ups_image":
        return [_cabi.plan_launch("spectrogram", *args, num_pad_frames=K, image_size=S, **kw),
                _cabi.plan_launch("synth", *args, num_pad_frames=K, **kw)]
    if r == "team":
        return [_cabi.plan_launch("spectrogram", *args, schedule=1, **kw), _cabi.plan_launch("debug", *args, **kw)]
    raise ValueError(r)


def _regimes(case):
    """the regimes a case's launches reach"""
    tags = set()
    T = case["T"]
    for p in _plans(case):
        sched = "team" if p["team"] else "coop"
        tags.add(sched)
        if p["team"]:
            tags.add("team-vm%d-nb%d" % (p["compiled_vm"], p["bodies_per_pass"]))
            if case.get("fma"):
                tags.add("team-fma")
            if p["ticket"]:
                tags.add("team-ticket")
            continue
        tags.add("coop-vm%d-nb%d" % (p["compiled_vm"], p["bodies_per_pass"]))
        tags.add("fma" if case.get("fma") else "planar")
        tags.add("ticket" if p["ticket"] else "grid=jobs")
        if not p["tma_loads"]:
            tags.add("no-tma-" + ("offset" if case.get("off") else "shape"))
        if p["ctas_per_sm"] == 1:
            tags.add("one-cta")
        if p["jobs_per_seq"] == 1 and p["tma_bulk_store"]:
            tags.add("bulk")
        if p["jobs_per_seq"] == 1 and p["tile_stride"] == 17 and p["columns_per_tile"] == 16 and not p["columns"] - p["columns_per_job"]:
            if -(-p["columns"] // 16) > 1:
                tags.add("rows17-subbatches")
        if p["jobs_per_seq"] == 1 and p["parked_sums"] and not case.get("K"):
            tags.add("park-one-job")
        if p["jobs_per_seq"] > 1 and p["parked_sums"] and not case.get("K") and p["columns"] > 0:
            tags.add("jobs")
            if p["z_capacity"] < 2304:
                tags.add("jobs-zcap<2304")
        if p["iq_fill"]:
            tags.add("iq-fill")
        if p["sparse_frames"]:
            tags.add("image-sparse")
        elif p["columns"] and case.get("S") and p["columns"] == case["S"]:
            tags.add("image-dense")
    if case.get("S"):
        tags.add("S=256" if case["S"] == 256 else "S!=256")
        tags.add("S%4" if case["S"] % 4 == 0 else "S-scalar")
    tags.add("T%%32=%d" % (T % 32))
    if T == 129:
        tags.add("T=129")
    tags.add("hop=%d" % case["hop"])
    E = len(case["edges"])
    if E in (1, 128):
        tags.add("E=%d" % E)
    for k in ("absent", "late", "radial", "offaxis", "ps", "views", "noise", "K"):
        if case.get(k):
            tags.add(k if k != "K" else "K=%d" % case["K"])
    tags.add("route-" + case["route"])
    from skeleton_action_recognition_b200 import _cabi
    src, dst = map(list, zip(*case["edges"]))
    grp = _cabi.partition_edges(src, dst, case["V"])
    if max(grp.count(g) for g in range(4)) >= 30:
        tags.add("group>=30")
    srcs = {}
    for s_, g in zip(src, grp):
        srcs.setdefault(g, set()).add(s_)
    if any(len(v) % 2 for v in srcs.values()):
        tags.add("odd-sources")
    if any(src.count(s_) > 1 for s_ in src):
        tags.add("multi-bone-joint")
    if len(set(case["edges"])) < E:
        tags.add("duplicate-bone")
    return tags


REQUIRED = {
    "coop", "team", "coop-vm50-nb2", "coop-vm0-nb1", "coop-vm0-nb2", "planar", "fma", "bulk", "rows17-subbatches",
    "park-one-job", "jobs", "jobs-zcap<2304", "no-tma-shape", "no-tma-offset", "one-cta", "grid=jobs", "ticket",
    "T=129", "T%32=0", "T%32=1", "T%32=31", "hop=8", "hop=16", "hop=37", "hop=100", "hop=200", "hop=300", "iq-fill",
    "E=1", "E=128", "group>=30", "odd-sources", "multi-bone-joint", "duplicate-bone", "absent", "late", "radial",
    "offaxis", "ps", "views", "noise", "K=3", "K=10", "route-synth", "route-ups_synth", "route-ups_debug",
    "route-ups_image", "route-image", "route-ready", "image-dense", "image-sparse", "S=256", "S!=256", "S%4", "S-scalar",
    "team-vm50-nb2", "team-vm0-nb1", "team-vm0-nb2", "team-fma", "team-ticket",
}


# ---- inputs ---------------------------------------------------------------------------------------------------------------
def _inputs(case, seed=0):
    """x (N / R, 3, T, V, M) float32, wavelengths (N,) and locations (N, 3) per output"""
    N, T, V, M = case["N"], case["T"], case["V"], case["M"]
    R = case.get("views", 1)
    g = torch.Generator().manual_seed(seed + 7 * T + V)
    Nx = N // R
    if case.get("radial"):
        dirs = torch.randn(Nx, 3, T, 1, M, generator=g)
        dirs = dirs / dirs.norm(dim=1, keepdim=True)
        r = 12 + 30 * torch.rand(Nx, 1, T, 1, M, generator=g)
        radial = dirs * (r + torch.arange(V).float().view(1, 1, 1, V, 1) * 0.25)
        x = torch.randn(Nx, 3, T, V, M, generator=g) * 0.3 + 15
        x[0, :, 300:420] = radial[0, :, 300:420]
        x[1, :, :, :, 1] = radial[1, :, :, :, 1]
    else:
        pose = torch.randn(Nx, 3, 1, V, M, generator=g) * 0.3
        t = torch.arange(T, dtype=torch.float32)[None, None, :, None, None]
        x = pose + 0.05 * torch.sin(2 * np.pi * 3 * t / 300 + torch.rand(Nx, 3, 1, V, M, generator=g) * 6.3)
        x = x + 0.01 * torch.randn(Nx, 3, T, V, M, generator=g)
    if case.get("absent") and M > 1:
        x[:, :, :, :, 1] = 0
    if case.get("late") and M > 1:
        x[:, :, case["late"]:, :, M - 1] = 0
    x = x.contiguous()
    lam = np.full(N, 1e-3, np.float32)
    loc = np.zeros((N, 3), np.float32)
    if case.get("offaxis"):
        loc[:] = [0.3, -0.2, 1.5]
    if case.get("ps"):
        lam = (1e-3 * (1 + 0.25 * np.arange(N))).astype(np.float32)
        loc[1::2] = np.array([0.3, -0.2, 1.5], np.float32) * (1 + np.arange(N)[1::2, None] * 0.1)
    return x, lam, loc


def _sentinel(shape):
    return torch.full(shape, SENTINEL, dtype=torch.int32, device="cuda").view(torch.float32)


def _no_sentinel(t):
    return int((t.view(torch.int32) == SENTINEL).sum())


# ---- stage 1: the float64 oracle and its bound ----------------------------------------------------------------------------
def _groups(src, dst, V):
    """per bone: (group, bones of its source joint, source joints of its group), and the largest group"""
    from skeleton_action_recognition_b200 import _cabi
    grp = np.array(_cabi.partition_edges(src, dst, V))
    nb = np.array([src.count(s) for s in src])
    ns = np.array([len({s for s, g in zip(src, grp) if g == grp[e]}) for e in range(len(src))])
    eg = max(int((grp == g).sum()) for g in range(4))
    return grp, nb, ns, eg


def bone_terms(pos, src, dst, lam, loc, mode):
    """float32 (theta (T, E, M), u, l) of every bone of one output (C recipes, the kernel's bits)"""
    p = torch.from_numpy(np.ascontiguousarray(pos[None]))
    S, D = p[:, :, :, src], p[:, :, :, dst]
    _, th = vro.range_phase_c(S, loc, float(lam), mode)
    u, ln = vro.aspect_cosine_c(S, D, loc, mode)
    return th[0].numpy(), u[0].numpy(), ln[0].numpy()


def stage1_oracle(th, u, ln, src, dst, V, u2_from=None, c_over=None, nan_rule=True):
    """z64 (T,), bound (T,), NaN mask (T,) from one output's float32 bone terms.  u2_from / c_over: wrong variants."""
    grp, nb, ns, eg = _groups(src, dst, V)
    E = len(src)
    M = th.shape[2]
    u64, l64, th64 = u.astype(np.float64), ln.astype(np.float64), th.astype(np.float64)
    u2 = u64 * u64 if u2_from is None else (u64 * u64)[:, u2_from]
    cbar = l64.sum(axis=1, keepdims=True) / (c_over or E)                 # (T, 1, M)
    c = cbar * cbar
    den = (1.0 - u2) + c * u2
    amp = np.sqrt(np.pi * c) / den
    z = (amp * np.exp(1j * th64)).sum(axis=(1, 2))
    eps_c = (eg + 4) * U
    dcm1 = 2 * c * eps_c + U * np.abs(c - 1)
    eps_den = (u2 * dcm1 + np.abs(c - 1) * U * u2 + U * den) / den
    kk = np.rint(th64 / (2 * np.pi))
    r = th64 - kk * 2 * np.pi
    dphi = np.abs(kk) * CW_ERR + U * np.abs(r)
    eps = (eps_den + RCP_REL + (nb[None, :, None] - 1) * U + eps_c + 2 * U + dphi + math.sqrt(2) * SINCOS_ABS
           + (ns[None, :, None] + M + 2) * U)
    bound = SAFETY * (np.abs(amp) * eps).sum(axis=(1, 2))
    nan = (u.astype(np.float32) * u.astype(np.float32) > 1).any(axis=(1, 2)) if nan_rule else np.zeros(len(z), bool)
    return z, bound, nan


def stage1_check(iq, z, bound, nan):
    """worst err/bound of the GPU's (or an emulation's) iq (T, 2) against the oracle; NaN exactly on the mask"""
    gn = np.isnan(iq[:, 0]) | np.isnan(iq[:, 1])
    assert np.array_equal(gn, nan), ("NaN mask", np.flatnonzero(gn != nan)[:10])
    ok = ~nan
    err = np.abs(iq[ok, 0].astype(np.float64) + 1j * iq[ok, 1].astype(np.float64) - z[ok])
    b = bound[ok]
    assert np.all(err[b == 0] == 0)
    return float((err / np.where(b > 0, b, 1.0)).max()) if err.size else 0.0


def stage1_output(pos_n, case, lam, loc, mode):
    src, dst = map(list, zip(*case["edges"]))
    th, u, ln = bone_terms(pos_n, src, dst, lam, loc, mode)
    return stage1_oracle(th, u, ln, src, dst, case["V"])


# ---- stage 2 --------------------------------------------------------------------------------------------------------------
def frame_index(frames, hop, T, pad="reflect", about=None):
    t = np.asarray(frames)[:, None] * hop - 128 + np.arange(256)[None, :]
    if pad == "edge":
        return np.clip(t, 0, T - 1)
    t = np.abs(t)
    return np.where(t >= T, 2 * ((T - 1) if about is None else about) - t, t)


def hann(symmetric=False):
    n = np.arange(256)
    return 0.5 - 0.5 * np.cos(2 * np.pi * n / (255 if symmetric else 256))


def stage2_oracle(iq, hop, frames=None, win=None, pad="reflect", shift=0, about=None, conj=False):
    """iq (T, 2) float32 -> |X| (256 bins, F), delta (F,) and the NaN mask (F,) of the listed frames (all by default).
    win / pad / shift / about / conj: wrong variants."""
    T = iq.shape[0]
    frames = np.arange(T // hop + 1) if frames is None else np.asarray(frames)
    z = iq[:, 0].astype(np.float64) + 1j * iq[:, 1].astype(np.float64)
    idx = frame_index(frames, hop, T, pad, about)
    if shift:
        idx = np.clip(frame_index(frames, hop, T) + shift, 0, T - 1)
    w = z[idx]
    nan = np.isnan(w).any(axis=1)
    w = np.where(np.isnan(w), 0, w)
    h = hann() if win is None else win
    hw = h[None, :] * w
    X = np.fft.ifft(hw, axis=1) * 256 if conj else np.fft.fft(hw, axis=1)
    delta = SAFETY * (GAMMA_FFT * np.abs(hw).sum(axis=1) + U * np.abs(w).sum(axis=1))
    return np.abs(X).T, delta, nan


def _eps_log(v):
    return SAFETY * (U + np.maximum(LOG_ABS, LOG_ULP * 2.0 ** -23 * np.abs(np.log(v))))


def stage2_check(out, A, delta, nan, roll=128):
    """worst err/bound of out (256, F) [rows fftshifted] against |X64| A (256 bins, F); NaN exactly on the frames' mask"""
    return _interval_ratio(np.roll(np.asarray(out, np.float64), -roll, axis=0), A, delta, nan)


def image_check(img, iq, hop, S):
    """the (S, S) image of one output against stage 2 of its I/Q: pixel (r, c) shows row rmap[r], frame fmap[c]"""
    T = iq.shape[0]
    fmap = resize.nearest_index(S, T // hop + 1)
    rmap = resize.nearest_index(S, 256)
    frames, inv = np.unique(fmap, return_inverse=True)
    A, delta, nan = stage2_oracle(iq, hop, frames)
    bins = (rmap - 128) % 256                                             # spectrogram row rmap[r] holds that bin
    return _interval_ratio(np.asarray(img, np.float64), A[:, inv][bins], delta[inv], nan[inv])


def _interval_ratio(o, A, delta, nan):
    """o (rows, F) against |X64| A of the same rows: the distance from ln(|X64| + 1e-6) over the distance to the interval's
    end on that side; NaN exactly on the frames' mask"""
    gn = np.isnan(o)
    want = np.broadcast_to(nan[None, :], o.shape)
    assert np.array_equal(gn, want), ("NaN mask", np.argwhere(gn != want)[:10])
    ok = ~want
    dp = delta[None, :] + SAFETY * (A + delta[None, :]) * (U + SQRT_REL)
    lo_v = np.maximum(A - dp, 0) + 1e-6 * (1 - U)
    hi_v = A + dp + 1e-6 * (1 + U)
    lo, hi, mid = np.log(lo_v) - _eps_log(lo_v), np.log(hi_v) + _eps_log(hi_v), np.log(A + 1e-6)
    d = o - mid
    r = np.where(d >= 0, d / (hi - mid), -d / (mid - lo))
    return float(r[ok].max()) if ok.any() else 0.0


# ---- CPU: pins ------------------------------------------------------------------------------------------------------------
def _cpu_case(seed=0, T=200, M=2, offaxis=True):
    g = torch.Generator().manual_seed(seed)
    x = (torch.randn(2, 3, T, 25, M, generator=g) * 0.3).contiguous()
    loc = np.array([0.3, -0.2, 1.5] if offaxis else [0, 0, 0], np.float32)
    return x, loc


def test_stage1_with_float64_terms_equals_the_hybrid_baseband():
    """stage 1's formula, fed float64 u, l and the float32 theta, is oracle.forward_hybrid's baseband to ~1e-12"""
    x, loc = _cpu_case()
    src, dst = map(list, zip(*NTU))
    xd = x.double()
    S, D = xd[:, :, :, src], xd[:, :, :, dst]
    L = torch.from_numpy(loc.astype(np.float64))[:, None, None, None]
    A, B = L - (S + D) / 2, D - S
    u = ((A * B).sum(1) / (A.norm(dim=1) * B.norm(dim=1) + 1e-6)).numpy()
    ln = B.norm(dim=1).numpy()
    lam32 = torch.tensor(1e-3, dtype=torch.float32)
    _, ph = vro.bone_geometry(x, src, dst, torch.from_numpy(loc), lam32, "seq")
    amp64, _ = vro.bone_geometry(xd, src, dst, torch.from_numpy(loc).double(), lam32.double())
    want = (amp64 * torch.exp(1j * ph.double())).sum(dim=(2, 3)).numpy()
    for n in range(2):
        z, _, _ = stage1_oracle(ph[n].numpy(), u[n], ln[n], src, dst, 25, nan_rule=False)
        assert np.abs(z - want[n]).max() <= 1e-12 * np.abs(want[n]).max()


def test_stage2_equals_the_float64_nnaudio_restatement():
    """stage 2's |X| is the float64 nnAudio restatement's to ~1e-12 of the peak, at hops below and above n_fft / 2"""
    g = torch.Generator().manual_seed(3)
    iq = torch.randn(2, 333, 2, generator=g)
    for hop in (16, 37, 200):
        o = vro.OracleVirtualRadar(hop_length=hop, dtype=torch.float64)
        want = vro.stft_logmag(iq.double(), o.stft, 256).numpy()
        for n in range(2):
            A, _, _ = stage2_oracle(iq[n].numpy(), hop)
            lin = np.exp(want[n]) - 1e-6                                    # |X| of the restatement, rows fftshifted
            assert np.abs(np.roll(A, 128, axis=0) - lin).max() <= 1e-12 * lin.max(), hop


# ---- CPU: a float32 emulation of the kernel, with every approximate instruction at its documented error ---------------------
f32 = np.float32


def _fma(a, b, c):
    return (np.asarray(a, np.float64) * np.asarray(b, np.float64) + np.asarray(c, np.float64)).astype(f32)


def emulate_synthesis(th, u, ln, src, dst, V, sign=1.0):
    """the kernel's float32 order of operations (bone_u2 -> joint_phase -> joints_pass -> team fold) on one output's
    float32 bone terms; rcp, __sincosf pushed by their documented error in the direction `sign`"""
    from skeleton_action_recognition_b200 import _cabi
    grp = np.array(_cabi.partition_edges(src, dst, V))
    T, E, M = th.shape
    inv_E = f32(1.0) / f32(E)
    u2 = (u * u).astype(f32)
    zg = np.zeros((4, T), np.complex128)
    for h in range(4):
        bones = [e for e in range(E) if grp[e] == h]
        joints = list(dict.fromkeys(src[e] for e in bones))
        zr = np.zeros(T, f32)
        zi = np.zeros(T, f32)
        for m in range(M):
            sums = []
            for hh in range(4):
                s = np.zeros(T, f32)
                for e in (e for e in range(E) if grp[e] == hh):
                    s = (s + ln[:, e, m]).astype(f32)
                sums.append(s)
            tot = ((sums[0] + sums[1]).astype(f32) + (sums[2] + sums[3]).astype(f32)).astype(f32)
            if not (tot != 0).any():
                continue
            cbar = (tot * inv_E).astype(f32)
            cm1 = _fma(cbar, cbar, -1.0)
            ar = np.zeros(T, f32)
            ai = np.zeros(T, f32)
            for j in joints:
                W = None
                for e in (e for e in bones if src[e] == j):
                    den = _fma(u2[:, e, m], cm1, 1.0)
                    w = ((1.0 / den.astype(np.float64)) * (1 + sign * RCP_REL)).astype(f32)
                    W = w if W is None else (W + w).astype(f32)
                e0 = next(e for e in bones if src[e] == j)
                t_ = th[:, e0, m]
                kk = ((_fma(t_, f32(0.15915494309189533577), f32(12582912.0)) - f32(12582912.0))).astype(f32)
                r = _fma(-kk, C1, t_)
                r = _fma(-kk, C2, r)
                cs = (np.cos(r.astype(np.float64)) + sign * SINCOS_ABS).astype(f32)
                sn = (np.sin(r.astype(np.float64)) + sign * SINCOS_ABS).astype(f32)
                ar = _fma(W, cs, ar)
                ai = _fma(W, sn, ai)
            K = (f32(1.7724538509055160273) * cbar).astype(f32)
            zr = _fma(K, ar, zr)
            zi = _fma(K, ai, zi)
        zg[h] = zr + 1j * zi
    re = ((zg[0].real.astype(f32) + zg[1].real.astype(f32)).astype(f32) + (zg[2].real.astype(f32) + zg[3].real.astype(f32)).astype(f32)).astype(f32)
    im = ((zg[0].imag.astype(f32) + zg[1].imag.astype(f32)).astype(f32) + (zg[2].imag.astype(f32) + zg[3].imag.astype(f32)).astype(f32)).astype(f32)
    nan = (u2 > 1).any(axis=(1, 2))
    iq = np.stack([re, im], axis=1)
    iq[nan] = np.nan
    return iq


def _padd(a, b):
    return ((a[0] + b[0]).astype(f32), (a[1] + b[1]).astype(f32))


def _psub(a, b):
    return ((a[0] - b[0]).astype(f32), (a[1] - b[1]).astype(f32))


def _pscale(a, r):
    return ((a[0] * r).astype(f32), (a[1] * r).astype(f32))


def _add_mj(a, b):
    return ((a[0] + b[1]).astype(f32), (a[1] - b[0]).astype(f32))


def _sub_mj(a, b):
    return ((a[0] - b[1]).astype(f32), (a[1] + b[0]).astype(f32))


def _pcmul(v, wx, wy):
    """v * (wx + j wy) as the kernel's FFMA2 / FMUL2 pair: (fma(v.y, -wy, v.x wx), fma(v.y, wx, v.x wy))"""
    return (_fma(v[1], -wy, (v[0] * wx).astype(f32)), _fma(v[1], wx, (v[0] * wy).astype(f32)))


def _dft4(x0, x1, x2, x3):
    t0, t1, t2, d = _padd(x0, x2), _psub(x0, x2), _padd(x1, x3), _psub(x1, x3)
    return _padd(t0, t2), _add_mj(t1, d), _psub(t0, t2), _sub_mj(t1, d)


def _dft8(v):
    R = f32(0.70710678118654752440)
    s = [_padd(v[i], v[i + 4]) for i in range(4)]
    d = [_psub(v[i], v[i + 4]) for i in range(4)]
    e1 = _pscale(_add_mj(d[1], d[1]), R)
    e3 = _pscale(_sub_mj(d[3], d[3]), -R)
    o = [None] * 8
    o[0], o[2], o[4], o[6] = _dft4(*s)
    t0, t1, t2, dd = _add_mj(d[0], d[2]), _sub_mj(d[0], d[2]), _padd(e1, e3), _psub(e1, e3)
    o[1], o[5], o[3], o[7] = _padd(t0, t2), _psub(t0, t2), _add_mj(t1, dd), _sub_mj(t1, dd)
    return o


def emulate_stft(iq, hop, sign=1.0):
    """stft_frame in float32, radix 8 x 8 x 4 in its butterfly order, every frame of one output -> out (256, F); the
    tables (cospif, sincospif), sqrt.approx and __logf pushed by their documented error in the direction `sign`"""
    T = iq.shape[0]
    F = T // hop + 1
    idx = frame_index(np.arange(F), hop, T)
    n = np.arange(256)
    cp = (np.cos(np.pi * (n * (2.0 / 256))) * (1 - sign * 2.0 ** -23)).astype(f32)
    h = _fma(f32(-0.5), cp, f32(0.5))
    zr, zi = iq[idx, 0].astype(f32), iq[idx, 1].astype(f32)                    # (F, 256)

    def tw(e):
        a = np.pi * ((e % 256) * (2.0 / 256))
        return (np.cos(a) * (1 + sign * 2.0 ** -24)).astype(f32), (-np.sin(a) * (1 + sign * 2.0 ** -24)).astype(f32)
    lane = np.arange(32)
    v = [_pscale((zr[:, lane + 32 * q], zi[:, lane + 32 * q]), h[lane + 32 * q]) for q in range(8)]
    v = _dft8(v)
    for q in range(1, 8):
        v[q] = _pcmul(v[q], *tw(lane * q))
    X1r = np.stack([a[0] for a in v], 1)                                       # (F, q, lane)
    X1i = np.stack([a[1] for a in v], 1)
    X1r, X1i = X1r.reshape(-1, 8, 8, 4), X1i.reshape(-1, 8, 8, 4)              # (F, k1, a, b4): lane = 4 a + b4
    v = [(X1r[:, :, a, :], X1i[:, :, a, :]) for a in range(8)]
    v = _dft8(v)
    b4 = np.arange(4)
    for c in range(1, 8):
        v[c] = _pcmul(v[c], *tw(8 * b4 * c))
    X2r = np.stack([a[0] for a in v], 2)                                       # (F, k1, c, b4)
    X2i = np.stack([a[1] for a in v], 2)
    out = np.zeros((F, 256), f32)
    for c in range(8):
        ys = _dft4(*[(X2r[:, :, c, b], X2i[:, :, c, b]) for b in range(4)])
        for d in range(4):
            kbin = np.arange(8) + 8 * c + 64 * d                               # k1 + 8 c + 64 d
            x, y = ys[d]
            m2 = _fma(x, x, (y * y).astype(f32))
            mag = (np.sqrt(m2.astype(np.float64)) * (1 + sign * SQRT_REL)).astype(f32)
            a = (mag + f32(1e-6)).astype(f32).astype(np.float64)
            lg = np.log(a)
            err = np.where((a >= 0.5) & (a <= 2), LOG_ABS, LOG_ULP * 2.0 ** -23 * np.abs(lg))
            out[:, (kbin + 128) % 256] = (lg + sign * err).astype(f32)
    return out.T


def _aligned_bones(seed=5, T=96):
    """positions with short bones (c ~ 1e-3) some of which point at the radar to within ~1e-4 rad (u ~ 1, den ~ c)"""
    g = np.random.default_rng(seed)
    V, M = 9, 2
    x = g.normal(0, 0.02, (3, T, V, M)).astype(np.float32) + np.array([0.4, -0.3, 2.0], np.float32)[:, None, None, None]
    loc = np.array([0.3, -0.2, 1.5], np.float32)
    for j in (1, 3, 5):
        d = x[:, :, j - 1, :] - loc[:, None, None]
        d = d / np.linalg.norm(d, axis=0, keepdims=True)
        jit = g.normal(0, 1e-4, d.shape)
        x[:, :, j, :] = (x[:, :, j - 1, :] + 0.03 * (d + jit)).astype(np.float32)
    edges = [(0, 1), (2, 3), (4, 5), (0, 6), (6, 7), (7, 8), (0, 2)]
    return x, loc, edges


@pytest.mark.parametrize("sign", [1.0, -1.0])
def test_criteria_accept_the_kernels_arithmetic(sign):
    """the emulation, approximate instructions at their documented error, passes both stages at err/bound <= 0.5"""
    x, loc, edges = _aligned_bones()
    src, dst = map(list, zip(*edges))
    worst1 = worst2 = 0.0
    for mode in ("seq", "fma"):
        th, u, ln = bone_terms(x, src, dst, 1e-3, loc, mode)
        assert (np.abs(u) > 0.9999).any() and not (u.astype(f32) * u.astype(f32) > 1).any()
        iq = emulate_synthesis(th, u, ln, src, dst, 9, sign)
        z, bound, nan = stage1_oracle(th, u, ln, src, dst, 9)
        worst1 = max(worst1, stage1_check(iq, z, bound, nan))
    x2, loc2 = _cpu_case(seed=1, T=333)
    th, u, ln = bone_terms(x2[0].numpy(), list(zip(*NTU))[0], list(zip(*NTU))[1], 1e-3, loc2, "seq")
    iq = emulate_synthesis(th, u, ln, list(zip(*NTU))[0], list(zip(*NTU))[1], 25, sign)
    z, bound, nan = stage1_oracle(th, u, ln, list(list(zip(*NTU))[0]), list(list(zip(*NTU))[1]), 25)
    worst1 = max(worst1, stage1_check(iq, z, bound, nan))
    for hop in (16, 37, 200):
        out = emulate_stft(iq, hop, sign)
        A, delta, nan2 = stage2_oracle(iq, hop)
        worst2 = max(worst2, stage2_check(out, A, delta, nan2))
    print("emulation err/bound: stage 1 %.3g, stage 2 %.3g" % (worst1, worst2))
    assert worst1 <= 0.5 and worst2 <= 0.5, (worst1, worst2)


def _reject(fn):
    try:
        r = fn()
    except AssertionError:
        return float("inf")
    return r


def test_criteria_reject_wrong_variants():
    x, loc = _cpu_case(seed=2, T=300)
    src, dst = map(list, zip(*NTU))
    th, u, ln = bone_terms(x[0].numpy(), src, dst, 1e-3, loc, "seq")
    z, bound, nan = stage1_oracle(th, u, ln, src, dst, 25)

    def as_iq(zz):
        return np.stack([zz.real, zz.imag], 1).astype(f32)
    shifted = z.copy()
    shifted[32] = z[33]                                                 # one sample shifted by a step at a chunk boundary
    variants1 = {
        "shifted sample": as_iq(shifted),
        "bone dropped": as_iq(stage1_oracle(th[:, 1:], u[:, 1:], ln[:, 1:], src[1:], dst[1:], 25, c_over=24)[0]),
        "body dropped": as_iq(stage1_oracle(th[:, :, :1], u[:, :, :1], ln[:, :, :1], src, dst, 25)[0]),
        "c over E - 1": as_iq(stage1_oracle(th, u, ln, src, dst, 25, c_over=23)[0]),
        "conjugated": as_iq(np.conj(z)),
        "u^2 of the neighbour": as_iq(stage1_oracle(th, u, ln, src, dst, 25, u2_from=np.roll(np.arange(24), 1))[0]),
    }
    good = as_iq(z)
    assert stage1_check(good, z, bound, nan) <= 0.5
    for name, iq in variants1.items():
        r = _reject(lambda: stage1_check(iq, z, bound, nan))
        assert r > 100, (name, r)
    iq = good
    T, hop = 300, 16
    A, delta, nan2 = stage2_oracle(iq, hop)

    def as_out(A_):
        return np.roll(np.log(A_ + 1e-6), 128, axis=0).astype(f32)
    assert stage2_check(as_out(A), A, delta, nan2) <= 0.5
    variants2 = {
        "symmetric Hann": as_out(stage2_oracle(iq, hop, win=hann(symmetric=True))[0]),
        "edge padding": as_out(stage2_oracle(iq, hop, pad="edge")[0]),
        "frame shifted by one": as_out(stage2_oracle(iq, hop, shift=1)[0]),
        "fftshift by 127": np.roll(np.log(A + 1e-6), 127, axis=0).astype(f32),
        "conjugated bins": as_out(stage2_oracle(iq, hop, conj=True)[0]),
        "last frame reflected about T - 2": as_out(stage2_oracle(iq, hop, about=T - 2)[0]),
    }
    for name, out in variants2.items():
        r = _reject(lambda: stage2_check(out, A, delta, nan2))
        assert r > 100, (name, r)


def test_case_table_reaches_every_regime():
    """through vr_plan_launch at 148 SMs: both schedules, every kernel instantiation family, store path and job regime"""
    import __graft_entry__ as ge
    ge.build()
    got = set()
    for c in CASES:
        got |= _regimes(c)
    assert REQUIRED <= got, sorted(REQUIRED - got)


# ---- GPU ------------------------------------------------------------------------------------------------------------------
def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _run(case, x, lam, loc):
    """launch the case's route with owned, sentinel-filled buffers -> dict of host arrays"""
    from skeleton_action_recognition_b200 import _cabi, pad_frames
    L = _cabi.lib()
    N, T, V, M, hop = case["N"], case["T"], case["V"], case["M"], case["hop"]
    src, dst = map(list, zip(*case["edges"]))
    sc, dc = _cabi.i32_array(src), _cabi.i32_array(dst)
    E = len(src)
    flags = _flags(case)
    ps = bool(flags & _cabi.VR_FLAG_PER_SEQUENCE)
    lam_d = torch.from_numpy(lam if ps else lam[:1]).cuda()
    loc_d = torch.from_numpy((loc if ps else loc[:1]).reshape(-1)).cuda()
    nx = x.numel()
    xbuf = torch.full((nx + 8,), float("nan"), device="cuda")
    o = 1 if case.get("off") else 0
    xbuf[o:o + nx] = x.reshape(-1).cuda()
    xp = xbuf.data_ptr() + 4 * o
    res = {}
    K = case.get("K", 0)
    Tu = T * K if K else T
    F = Tu // hop + 1
    st = _stream()
    noise = None
    if case.get("noise"):
        noise = (torch.tensor([0.0, 0.05, 1.0][:N] + [0.02] * max(0, N - 3), dtype=torch.float32, device="cuda"),
                 torch.tensor(12345, dtype=torch.int64, device="cuda"))

    def set_noise():
        if noise is not None:
            _cabi.set_noise(*noise)
    args = (xp, N, T, V, M, sc, dc, E, lam_d.data_ptr(), loc_d.data_ptr())
    r = case["route"]
    if K:
        nbytes = int(L.vr_upsampled_workspace_bytes(N // case.get("views", 1), T, V, M))
        work = torch.empty(nbytes // 8, dtype=torch.float64, device="cuda")
        res["pos"] = pad_frames(x.cuda(), K, 3.0).cpu().numpy()
    if r in ("debug", "ready", "team"):
        out, iq = _sentinel((N, 256, F)), _sentinel((N, T, 2))
        set_noise()
        _cabi.check(L.vr_forward_debug_f32(*args, 256, hop, flags, out.data_ptr(), iq.data_ptr(), st))
        if r == "ready":                                   # a second batch right behind, its reads not waiting for the first
            x2 = (x * 1.3 + 0.1).contiguous().cuda()
            out2, iq2 = _sentinel((N, 256, F)), _sentinel((N, T, 2))
            _cabi.check(L.vr_forward_debug_f32(x2.data_ptr(), *args[1:], 256, hop, flags, out2.data_ptr(), iq2.data_ptr(), st))
            res["out2"], res["iq2"], res["x2"] = out2, iq2, x2.cpu()
        res["out"], res["iq"] = out, iq
        if r == "team":
            out_t = _sentinel((N, 256, F))
            _cabi.set_schedule(1)
            try:
                _cabi.check(L.vr_forward_f32(*args, 256, hop, flags, out_t.data_ptr(), st))
            finally:
                _cabi.set_schedule(-1)
            res["out"] = out_t
    elif r == "synth":
        iq = _sentinel((N, T, 2))
        _cabi.check(L.vr_synth_f32(*args, flags, iq.data_ptr(), st))
        res["iq"] = iq
    elif r == "image":
        S = case["S"]
        img, iq = _sentinel((N, S, S)), _sentinel((N, T, 2))
        _cabi.check(L.vr_forward_image_f32(*args, 256, hop, flags, S, img.data_ptr(), st))
        _cabi.check(L.vr_synth_f32(*args, flags, iq.data_ptr(), st))
        res["img"], res["iq"] = img, iq
    elif r == "ups_debug":
        out, iq = _sentinel((N, 256, F)), _sentinel((N, Tu, 2))
        _cabi.check(L.vr_forward_upsampled_debug_f32(*args, 256, hop, flags, K, ctypes.c_float(3.0), work.data_ptr(), nbytes,
                                                     out.data_ptr(), iq.data_ptr(), st))
        res["out"], res["iq"] = out, iq
        synth = _sentinel((N, Tu, 2))
        _cabi.check(L.vr_synth_upsampled_f32(*args, flags, K, ctypes.c_float(3.0), work.data_ptr(), nbytes, synth.data_ptr(), st))
        res["synth"] = synth
    elif r == "ups_synth":
        iq = _sentinel((N, Tu, 2))
        _cabi.check(L.vr_synth_upsampled_f32(*args, flags, K, ctypes.c_float(3.0), work.data_ptr(), nbytes, iq.data_ptr(), st))
        res["iq"] = iq
    elif r == "ups_image":
        S = case["S"]
        img, iq = _sentinel((N, S, S)), _sentinel((N, Tu, 2))
        _cabi.check(L.vr_forward_upsampled_f32(*args, 256, hop, flags, K, ctypes.c_float(3.0), S, work.data_ptr(), nbytes,
                                               img.data_ptr(), st))
        _cabi.check(L.vr_synth_upsampled_f32(*args, flags, K, ctypes.c_float(3.0), work.data_ptr(), nbytes, iq.data_ptr(), st))
        res["img"], res["iq"] = img, iq
    if r in ("debug", "ready") or r == "ups_debug":
        synth = res.get("synth")
        if synth is None:
            synth = _sentinel((N, Tu, 2))
            set_noise()
            _cabi.check(L.vr_synth_f32(*args, flags, synth.data_ptr(), st))
        res["synth"] = synth
    torch.cuda.synchronize()
    for k, v in list(res.items()):
        if isinstance(v, torch.Tensor) and v.is_cuda:
            assert _no_sentinel(v) == 0, (case["id"], k, "unwritten entries", _no_sentinel(v))
            res[k] = v.cpu().numpy()
        elif isinstance(v, torch.Tensor):
            res[k] = v.numpy()
    return res


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c["id"] for c in CASES])
def test_fused_forward_stage_by_stage(case):
    x, lam, loc = _inputs(case)
    res = _run(case, x, lam, loc)
    mode = "fma" if case.get("fma") else "seq"
    R = case.get("views", 1)
    hop, N = case["hop"], case["N"]
    if "synth" in res and "out" in res and case["route"] != "team":      # debug I/Q = synthesis-only I/Q, every sample
        assert np.array_equal(res["iq"].view(np.int32), res["synth"].view(np.int32)), case["id"]
    w1 = w2 = 0.0
    xs = [(res.get("pos", x.numpy()), res["iq"], "out")]
    if case["route"] == "ready":
        xs.append((res["x2"], res["iq2"], "out2"))
    for pos, iq, okey in xs:
        for n in range(N):
            if not case.get("noise") and case["route"] != "team":
                z, bound, nan = stage1_output(pos[n // R], case, lam[n], loc[n], mode)
                w1 = max(w1, stage1_check(iq[n], z, bound, nan))
            if "img" in res:
                w2 = max(w2, image_check(res["img"][n], iq[n], hop, case["S"]))
            elif okey in res:
                A, delta, nan2 = stage2_oracle(iq[n], hop)
                w2 = max(w2, stage2_check(res[okey][n], A, delta, nan2))
    print("%s: stage 1 err/bound %.3g, stage 2 err/bound %.3g" % (case["id"], w1, w2))
    assert w1 <= 1 and w2 <= 1, (case["id"], w1, w2)
