"""TEST INFRASTRUCTURE ONLY -- gradients of the VirtualRadar layer with respect to `wavelength` and
`radar_location` (reference layers/virtual_radar.py:40-41, 65-69: trainable nn.Parameters; the reference
obtains the gradients from PyTorch autograd over forward(), :79-134).

Two independent routes, both on the CPU:
  autograd_grads   the oracle's own torch graph (oracle/virtual_radar_oracle.py, the reference's ops in the
                   reference's order) differentiated by torch.autograd, in float64 ("truth") or float32 (what
                   the reference itself would return).
  analytic_grads   the closed form the CUDA kernels implement (csrc/vr_backward.cuh), written with numpy in
                   float64: adjoint of the windowed STFT + log magnitude, then the derivatives of
                   z = sum amp * exp(j theta).  tests/test_oracle.py pins it to autograd_grads.
  synth_adjoint    the second stage alone (dL/d(iq) -> parameter and skeleton gradients) with the CUDA kernel's
                   deliberate roundings: float32 range, phase and mean bone length, float64 everything else, in the
                   kernel's order of operations.  It returns each path of the gradient separately, and the sums of
                   absolute terms from which tests/test_backward_property_gpu.py derives its tolerances.
"""
import numpy as np
import torch

from . import virtual_radar_oracle as vro


def autograd_grads(x, grad_out, edges=vro.NTU_EDGES, wavelength=1e-3, radar_location=(0., 0., 0.),
                   n_fft=256, hop_length=16, dtype=torch.float64, wrt_x=False):
    """-> (dL/dwavelength, dL/dradar_location, out) or, with wrt_x, (.., .., dL/dx)."""
    o = vro.OracleVirtualRadar(edges, wavelength, radar_location, n_fft, hop_length, dtype)
    lam = o.wavelength.clone().requires_grad_(True)
    loc = o.radar_location.clone().requires_grad_(True)
    xx = x.to(dtype).clone().requires_grad_(wrt_x)
    iq = vro.synthesize_iq(xx, o.src, o.dst, loc, lam, "aten")
    out = vro.stft_logmag(iq, o.stft, n_fft)
    loss = (out * torch.as_tensor(grad_out).to(dtype)).sum()
    grads = torch.autograd.grad(loss, (lam, loc, xx) if wrt_x else (lam, loc))
    if wrt_x:
        return float(grads[0]), grads[1].numpy().astype(np.float64), grads[2].numpy().astype(np.float64)
    return float(grads[0]), grads[1].numpy().astype(np.float64), out.detach().numpy()


def _reflect(t, T):
    t = np.abs(t)
    return np.where(t >= T, 2 * (T - 1) - t, t)


def stft_adjoint(iq, grad_out, n_fft=256, hop=16):
    """iq (N,T,2), grad_out (N,n_fft,F) -> dL/d(iq) (N,T,2), float64."""
    iq = np.asarray(iq, np.float64)
    g = np.asarray(grad_out, np.float64)
    N, T, _ = iq.shape
    F = T // hop + 1
    z = iq[..., 0] + 1j * iq[..., 1]
    n = np.arange(n_fft)
    w = 0.5 - 0.5 * np.cos(2 * np.pi * n / n_fft)
    gz = np.zeros((N, T), np.complex128)
    for f in range(F):
        idx = _reflect(f * hop - n_fft // 2 + n, T)
        X = np.fft.fft(z[:, idx] * w, axis=1)                     # X[k] = sum w zp e^{-j 2 pi k n / n_fft}
        a = np.abs(X)
        gk = np.roll(g[:, :, f], -(n_fft // 2), axis=1)           # out row r shows bin (r - n_fft/2) mod n_fft
        G = np.where(a > 0, gk * X / (a * (a + 1e-6) + (a == 0)), 0)
        y = w * (np.fft.ifft(G, axis=1) * n_fft)                  # sum_k G e^{+j 2 pi k n / n_fft}
        np.add.at(gz, (slice(None), idx), y)
    return np.stack((gz.real, gz.imag), -1)


def analytic_grads(x, grad_out, edges=vro.NTU_EDGES, wavelength=1e-3, radar_location=(0., 0., 0.),
                   n_fft=256, hop_length=16, wrt_x=False):
    x64 = np.asarray(x, np.float64)
    lam = float(np.float32(wavelength))
    L = np.asarray(np.float32(radar_location), np.float64)[None, :, None, None, None]
    src, dst = map(list, zip(*edges))
    S, D = x64[:, :, :, src], x64[:, :, :, dst]                  # (N,3,T,E,M)
    rng = np.sqrt(((S - L) ** 2).sum(1))
    th = 4 * np.pi * rng / lam
    A, B = L - (S + D) / 2, D - S
    na, nb = np.sqrt((A ** 2).sum(1)), np.sqrt((B ** 2).sum(1))
    dot = (A * B).sum(1)
    q = na * nb + 1e-6
    u = dot / q
    cbar = nb.mean(axis=2, keepdims=True)
    c = cbar ** 2
    K = np.sqrt(np.pi) * cbar
    den = 1 + (c - 1) * u ** 2
    amp = K / den
    iq = np.stack(((amp * np.cos(th)).sum((2, 3)), (amp * np.sin(th)).sum((2, 3))), -1)
    gz = stft_adjoint(iq, grad_out, n_fft, hop_length)
    gI, gQ = gz[..., 0][:, :, None, None], gz[..., 1][:, :, None, None]
    dth = amp * (gQ * np.cos(th) - gI * np.sin(th))
    damp = gI * np.cos(th) + gQ * np.sin(th)
    g_lam = (dth * (-th / lam)).sum()
    with np.errstate(divide="ignore", invalid="ignore"):
        kth = np.where(rng > 0, dth * (4 * np.pi / lam) / rng, 0)[:, None]
        kamp = (damp * (-K * 2 * u * (c - 1) / den ** 2))[:, None]
        dudA = np.where(na[:, None] > 0, B / q[:, None] - (dot * nb / (na * q ** 2))[:, None] * A, 0)
    g_loc = (kth * (L - S) + kamp * dudA).sum((0, 2, 3, 4))
    if not wrt_x:
        return float(g_lam), g_loc, iq
    # dL/dx: through the range (S), the aspect cosine (A = L - (S+D)/2, B = D - S) and the mean bone length
    with np.errstate(divide="ignore", invalid="ignore"):
        dudB = np.where(nb[:, None] > 0, A / q[:, None] - (dot * na / (nb * q ** 2))[:, None] * B, 0)
        unitB = np.where(nb[:, None] > 0, B / nb[:, None], 0)
    G_c = (damp * np.sqrt(np.pi) * (1 / den - 2 * c * u ** 2 / den ** 2)).sum(2, keepdims=True)     # (N,T,1,M)
    gB = kamp * dudB + (G_c / len(src))[:, None] * unitB
    gS = kth * (S - L) - 0.5 * kamp * dudA - gB
    gD = -0.5 * kamp * dudA + gB
    gx = np.zeros_like(x64)
    for e, (si, di) in enumerate(zip(src, dst)):
        gx[:, :, :, si] += gS[:, :, :, e]
        gx[:, :, :, di] += gD[:, :, :, e]
    return float(g_lam), g_loc, gx


PATHS = ("phase", "u", "length")


def _bone_lengths_f32(S, D, mode):
    """|D - S| of every bone in float32 as the kernel rounds it: float32 B = D - S, norm in the layout's mode."""
    loc0 = np.zeros(3, np.float32)
    _, ln = vro.aspect_cosine_c(torch.from_numpy(np.ascontiguousarray(S)), torch.from_numpy(np.ascontiguousarray(D)),
                                loc0, mode)
    return ln.numpy()


def synth_adjoint(x, giq, edges=vro.NTU_EDGES, wavelength=1e-3, radar_location=(0., 0., 0.), mode="seq",
                  theta32=True, cbar32=True):
    """The synthesis adjoint of csrc/vr_backward.cuh (synth_adjoint_body) in numpy.

    x (N,3,T,V,M) float32, giq = dL/d(iq) (N,T,2), mode "seq" / "fma": the range rounding of the layout
    (VR_FLAG_RANGE_FMA).  Roundings as in the kernel:
      * range d and phase theta: float32, bit-exact (range_phase_c), unless theta32=False (float64 norm and phase);
      * mean bone length: float32 B = D - S, norm in `mode`, float32 sum in edge order, times f32(1/E), unless
        cbar32=False (float64 mean; the derivative then uses 1/E instead of f32(1/E));
      * the aspect cosine u, the amplitude and every derivative: float64 from the float32 inputs, in the kernel's order
        of operations, with its guards (d > 0, |A| > 0, |B| > 0) and the absent-body rule (float32 sum of the bone
        lengths == 0: the body contributes exactly 0).  A time step whose dL/d(iq) is exactly 0 contributes 0.

    Returns a dict, all float64:
      "lam", "loc" (3,), "x" (N,3,T,V,M)   the gradients;
      "paths"[p][k]                          the part of gradient k ("lam", "loc", "x") through path p: "phase" (the
                                             range d), "u" (the aspect cosine), "length" (the mean bone length);
      "scale"[p][k]                          the sum of |term| of path p: per parameter over all (sequence, step,
                                             bone, body) terms, per dL/dx entry over the bones that touch it.
    """
    x = np.asarray(x, np.float32)
    g = np.asarray(giq, np.float64)
    N, _, T, V, M = x.shape
    src, dst = map(list, zip(*edges))
    E = len(src)
    lam32 = np.float32(wavelength)
    lam = float(lam32)
    loc32 = np.asarray(radar_location, np.float32)
    L = loc32.astype(np.float64)[:, None, None, None]
    inv_E = float(np.float32(1) / np.float32(E)) if cbar32 else 1.0 / E
    PI = np.pi
    sqrt_pi = np.sqrt(PI)
    zeros = lambda *s: np.zeros(s)                                              # noqa: E731
    out = {"paths": {p: {"lam": 0.0, "loc": zeros(3), "x": zeros(*x.shape)} for p in PATHS},
           "scale": {p: {"lam": 0.0, "loc": zeros(3), "x": zeros(*x.shape)} for p in PATHS}}
    for n in range(N):
        S32, D32 = x[n][:, :, src], x[n][:, :, dst]                             # (3,T,E,M)
        if theta32:
            d, th = vro.range_phase_c(torch.from_numpy(S32[None]), loc32, lam32, mode)
            rng, th = d.numpy()[0].astype(np.float64), th.numpy()[0].astype(np.float64)
        else:
            rng = np.sqrt(((S32.astype(np.float64) - L) ** 2).sum(0))
            th = 4 * PI * rng / lam
        if cbar32:
            ln = _bone_lengths_f32(S32[None], D32[None], mode)[0]               # (T,E,M) float32
            sumB = np.zeros((T, M), np.float32)
            for e in range(E):
                sumB = sumB + ln[:, e]
            cbar = (sumB * np.float32(inv_E)).astype(np.float64)[:, None]       # (T,1,M)
            absent = (sumB == 0)[:, None]
        else:
            nb64 = np.sqrt(((D32.astype(np.float64) - S32) ** 2).sum(0))
            cbar = nb64.sum(1, keepdims=True) * inv_E
            absent = cbar == 0
        gI, gQ = g[n, :, 0][:, None, None], g[n, :, 1][:, None, None]
        active = ~absent & ~((gI == 0) & (gQ == 0))                             # (T,E or 1,M)
        S, D = S32.astype(np.float64), D32.astype(np.float64)
        c = cbar * cbar
        K = sqrt_pi * cbar
        sn, cs = np.sin(th), np.cos(th)
        B = D - S
        A = L - 0.5 * (S + D)
        na = np.sqrt(A[0] * A[0] + A[1] * A[1] + A[2] * A[2])
        nb = np.sqrt(B[0] * B[0] + B[1] * B[1] + B[2] * B[2])
        dot = A[0] * B[0] + A[1] * B[1] + A[2] * B[2]
        q = na * nb + 1e-6
        u = dot / q
        den = 1.0 + (c - 1.0) * u * u
        amp = K / den
        dth = amp * (gQ * cs - gI * sn)
        damp = gI * cs + gQ * sn
        with np.errstate(divide="ignore", invalid="ignore"):
            t_lam = np.where(active, dth * (-th / lam), 0)
            kth = np.where(active & (rng > 0), dth * (4.0 * PI / lam) / rng, 0)
            kamp = np.where(active, damp * (-K * 2.0 * u * (c - 1.0) / (den * den)), 0)
            r2 = dot * nb / (na * q * q)
            dA = np.where(na > 0, kamp * (B / q - r2 * A), 0)                   # dL/dA through u
            r3 = dot * na / (nb * q * q)
            dB = np.where(nb > 0, kamp * (A / q - r3 * B), 0)                   # dL/dB through u
            G_c = np.where(active, damp * sqrt_pi * (1.0 / den - 2.0 * c * u * u / (den * den)), 0).sum(1, keepdims=True)
            kc = np.where(nb > 0, G_c * inv_E / nb, 0)
        ph_loc = kth * (L - S)
        # per bone: (dL/dS, dL/dD) of each path
        parts = {"phase": (kth * (S - L), np.zeros_like(S)),
                 "u": (-0.5 * dA - dB, -0.5 * dA + dB),
                 "length": (-kc * B, kc * B)}
        P, C = out["paths"], out["scale"]
        P["phase"]["lam"] += t_lam.sum()
        C["phase"]["lam"] += np.abs(t_lam).sum()
        P["phase"]["loc"] += ph_loc.sum((1, 2, 3))
        C["phase"]["loc"] += np.abs(ph_loc).sum((1, 2, 3))
        P["u"]["loc"] += dA.sum((1, 2, 3))
        C["u"]["loc"] += np.abs(dA).sum((1, 2, 3))
        for p, (gS, gD) in parts.items():
            px, cx = P[p]["x"][n], C[p]["x"][n]
            for e, (si, di) in enumerate(zip(src, dst)):
                px[:, :, si] += gS[:, :, e]
                px[:, :, di] += gD[:, :, e]
                cx[:, :, si] += np.abs(gS[:, :, e])
                cx[:, :, di] += np.abs(gD[:, :, e])
    for k in ("lam", "loc", "x"):
        out[k] = sum(out["paths"][p][k] for p in PATHS)
    return out
