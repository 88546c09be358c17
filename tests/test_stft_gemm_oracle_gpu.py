"""The general-kernel STFT (csrc/vr_stft_gemm.cuh behind vr_stft_general_f32, vr_stft_general_frames_f32 and their backward
passes) stage by stage against float64, in every launch regime of its host plan (vr_plan_stft_general).

Each stage is compared with float64 computed from THAT stage's float32 inputs as the GPU left them (the test owns every
buffer and reads every intermediate back), with a bound per entry.  So the ill-conditioning of d ln|X| at |X| ~ 0, which
forces the end-to-end gradient tests to aggregate bars, enters no comparison here, and a misplaced row, bin, frame, K
block or split slice is an error of order one against a bound near 1e-5.

The float64 oracle is written from the definition, in natural order (never through the kernel's tiled Bt):

    Re[m, b] = sum_j I_m[j] wcos[b, j] + Q_m[j] wsin[b, j]       Im[m, b] = sum_j Q_m[j] wcos[b, j] - I_m[j] wsin[b, j]

with frame m = (sequence s, frame f), I_m[j] = frames_work[s, 0, f hop' + j] (hop' = hop, or n_fft for the kept route's
compact copy), and its transposes: dA = dL/d(frame) (row m, columns [I | Q]), dL/dwcos = sum_m dRe I + dIm Q,
dL/dwsin = sum_m dRe Q - dIm I.  Two white-box layouts are restated from vr_stft_gemm.cuh: the tiled column order of
c_save / dc_work (stft_row_re / stft_row_im, nb = min(n_fft, 64) bins per column tile: [Re of nb bins | Im of them]) and
their column-major storage with leading dimension ldm (vr_stft_dc_kernel, the forward epilogue).

The bound gamma(K) of one GEMM entry, relative to S = sum_k |a_k b_k| of that entry (DESIGN 3d, the 3-term TF32 split):

    a = hi + lo, hi = a rounded to TF32 (11 significant bits), |lo| <= 2^-11 |a|; three MMAs per K step.
    (1) the dropped lo.lo term                                    |lo_a lo_b| <= 2^-22 |a b|
    (2) lo enters the tensor core as TF32 (13 of its bits cut),
        in each of the two cross terms                            <= 2^-10 |lo| |hi| <= 2^-21 |a b|, twice
    (3) one truncation per MMA instruction into its accumulator, whose value is bounded by the partial S: the hi.hi
        products take K/8 instructions (rotating over three accumulators)                       <= (K/8) 2^-23 S
    (4) the products' alignment inside one instruction, counted once more                      <= (K/8) 2^-23 S
    (5) the cross-term accumulator: 2 K/8 truncations of a value <= 2^-10 S                    <= (2K/8) 2^-33 S
    (6) the epilogue's three float32 adds of the four accumulators                             <= 3 2^-24 S
    gamma(K) = SAFETY (2^-22 + 2^-20 + (K/4) 2^-23 + (K/4) 2^-33 + 3 2^-24),  K rounded up to whole 32-column K blocks

SAFETY = 2 covers the second-order terms the list drops (products of the 2^-11 and 2^-23 factors, partial sums of |hi b|
exceeding S by (1 + 2^-11)^2).  The kernel gradient is `splits` such GEMMs over kb_per_split K blocks each, whose partial
planes are added in slice order (splits - 1 float32 adds) and then combined by one more add (dL/dwcos = dBt[re] + dBt[im]):
gamma_dBt = gamma(32 kb_per_split) + SAFETY splits 2^-24, against S over all M frames.

Criteria per stage (each GPU case prints the worst err/bound of each):

  pad / gather   frames_work bit-equal to numpy's reflect padding (nnAudio center=True), zeros in [T + n_fft, Lp); the kept
                 route's compact copy bit-equal to the listed frames of it
  forward        c_save within gamma(2 n_fft) S per entry
  epilogue       out[s, (b + n/2) % n, f] = ln(sqrt(re^2 + im^2) + 1e-6) of the GPU's own c_save within 4 ulp + 2^-22
                 (argument: 2 roundings in the square sum, sqrt, the add: <= 3 2^-24 relative, i.e. absolute after the
                 log; logf <= 1 ulp plus its rounding)
  dc             within 16 2^-24 |ref| of float64 from the GPU's c_save and grad_out (7 roundings: im*im, fma, sqrt, + 1e-6,
                 the product, the division, the scaling); exactly 0 where |X| = 0 (float64 autograd gives NaN there: a
                 deliberate difference, pinned on the CPU) and in the padding rows M .. ldm
  dA             within gamma(2 n_fft) S per entry, from the GPU's dc_work
  fold           (number of terms) 2^-24 sum|terms| per sample, from the GPU's da_work; exactly 0 where no frame (no kept
                 frame) covers the sample
  dBt + dw       within gamma_dBt S per entry, from the GPU's dc_work and frames_work

The CPU tests pin the oracle to `_STFTKernels._logmag_torch` and to oracle/nnaudio_stft.py in float64 (and its backward
to float64 autograd), show that the same checkers accept the float64 oracle rounded to float32 and reject seven
deliberately wrong variants, and check that the case table reaches every regime of the host plan at 148 SMs."""
import ctypes

import numpy as np
import pytest
import torch

U24 = 2.0 ** -24
SAFETY = 2.0
SMS = 148

# ---- the case table -----------------------------------------------------------------------------------------------------
# (N, T, n_fft, hop, kept frames, buffers offset from their 16-byte alignment, first sequence all zero)
#   kept frames: None = the full route; ("resize", S) = kept_frame_table(T // hop + 1, S); ("ends",) = first and last frame;
#   a tuple = those frame indices.  Offsets: "frames" (frames_work + 1 float), "da" / "dbt" (da_work / dbt_work + 1 float:
#   scalar EPI-0 stores), "iq" / "giq" (iq / grad_iq + 8 bytes) -- all legal under the header's alignment contract.
CASES = [
    (1, 2050, 256, 16, None, ("frames",), False),       # M = 129 = 1 (mod 128, 32): a ragged row tile of one row; T % 4 = 2
    #                                                     (Lp padded); 5 K blocks unsplit; unaligned frame rows at hop % 4 = 0
    (3, 40, 32, 50, None, ("iq", "giq"), False),        # F = 1 (hop > T); hop > n_fft, hop % 4 != 0: samples 17..39 uncovered
    (1, 9, 16, 3, None, (), False),                     # the shortest T = n_fft/2 + 1: the reflected margins cover the whole
    #                                                     signal; 32 of the one column tile's 128 rows valid
    (1, 1600, 64, 1, None, (), False),                  # M = 1601: 7 split-K slices of 8 K blocks, the last of 3; hop = 1
    (435, 130, 256, 27, None, ("da",), False),          # M = 2175 = 127 (mod 128), 31 (mod 32); F = 5; 16 kernel-gradient
    #                                                     tiles x 9 slices, the last of 4
    (2, 1500, 1024, 128, None, ("da", "dbt"), False),   # 16 column tiles x 64 K blocks; 256 kernel-gradient tiles: more CTAs
    #                                                     than SMs, unsplit, scalar stores
    (1, 3073, 512, 4, None, ("frames",), False),        # M = 769 = 1 (mod 128): 64 tiles x 2 slices of 13 and 12 K blocks
    (2, 1020, 128, 8, None, ("dbt",), False),           # M = 256 = 0 (mod 128); 4 tiles, one slice of 8 K blocks
    (18, 40, 64, 32, None, ("da", "dbt"), True),        # F = 2, M = 36 = 4 (mod 32): frame chunks cross sequences; |X| = 0
    (53, 50, 32, 20, None, (), False),                  # F = 3, M = 159 = 31 (mod 32)
    (4, 301, 16, 37, None, ("iq",), False),             # hop > n_fft with F = 9: gaps between frames; T % 4 = 1
    (2, 3000, 64, 8, ("resize", 100), ("frames", "giq"), False),   # kept: nearest resize of 376 frames to 100; 7 K blocks
    (3, 300, 128, 16, (7,), (), False),                 # kept: a single frame
    (5, 203, 32, 6, ("ends",), (), False),              # kept: the first and last frames only; hop % 4 != 0
    (30, 2000, 256, 16, (0, 3, 40, 41, 90, 125), ("da",), True),   # kept: gaps up to 49 frames > n_fft / hop = 16; 6 K blocks
]


def case_id(c):
    N, T, n, hop, kept, off, zero = c
    k = "" if kept is None else "-kept%s" % ("".join(str(v) for v in kept) if kept[0] in ("resize", "ends") else len(kept))
    return "N%d-T%d-n%d-h%d%s%s%s" % (N, T, n, hop, k, "".join("-" + o for o in off), "-zero" if zero else "")


def kept_frames(case):
    """int32 frame table of a case (None: the full route)."""
    N, T, n, hop, kept = case[:5]
    if kept is None:
        return None
    F = T // hop + 1
    if kept[0] == "resize":
        from skeleton_action_recognition_b200.layers.virtual_radar import kept_frame_table
        return kept_frame_table(F, kept[1])
    if kept[0] == "ends":
        return np.array([0, F - 1], dtype=np.int32)
    return np.array(kept, dtype=np.int32)


# ---- white-box layouts, restated from vr_stft_gemm.cuh (stft_row_re / stft_row_im; c_save and dc_work column-major) ----
def tiled_columns(n_fft):
    nb = min(n_fft, 64)
    b = np.arange(n_fft)
    re = (b // nb) * 2 * nb + b % nb
    return re, re + nb


def read_columns(buf, n_fft, ldm, M):
    """c_save / dc_work -> (Re (M, n_fft), Im (M, n_fft)) in bin order."""
    C = np.asarray(buf[:2 * n_fft * ldm]).reshape(2 * n_fft, ldm)
    re, im = tiled_columns(n_fft)
    return C[re, :M].T, C[im, :M].T


# ---- the float64 oracle -----------------------------------------------------------------------------------------------
def reflect(u, T, n_fft):
    """sample index held at padded position u (nnAudio center=True, pad_mode='reflect')"""
    t = np.abs(np.asarray(u) - n_fft // 2)
    return np.where(t >= T, 2 * (T - 1) - t, t)


def pad_oracle(iq, n_fft, Lp):
    """iq (N, T, 2) -> the planar padded signal (N, 2, Lp) the full route's frame views read; zeros past T + n_fft."""
    N, T, _ = iq.shape
    P = np.zeros((N, 2, Lp), dtype=iq.dtype)
    P[:, :, :T + n_fft] = np.pad(iq.transpose(0, 2, 1), ((0, 0), (0, 0), (n_fft // 2, n_fft // 2)), mode="reflect")
    return P


def gather_oracle(iq, frames, n_fft, hop):
    """the kept route's compact copy (N, 2, F_kept n_fft): the listed frames of the padded signal end to end"""
    P = pad_oracle(iq, n_fft, iq.shape[1] + n_fft)
    idx = (np.asarray(frames, dtype=np.int64)[:, None] * hop + np.arange(n_fft)).ravel()
    return P[:, :, idx]


def frame_rows(P, F, n_fft, hop_view):
    """planar signal (N, 2, Lp) -> I, Q frame matrices (N F, n_fft) in float64"""
    N = P.shape[0]
    idx = np.arange(F)[:, None] * hop_view + np.arange(n_fft)
    X = np.asarray(P, dtype=np.float64)[:, :, idx]                       # (N, 2, F, n)
    return X[:, 0].reshape(N * F, n_fft), X[:, 1].reshape(N * F, n_fft)


def forward_oracle(I, Q, wsin, wcos):
    """Re, Im (M, n_fft) and the abs-sums S of every entry"""
    ws, wc = np.asarray(wsin, np.float64).reshape(wsin.shape[0], -1), np.asarray(wcos, np.float64).reshape(wcos.shape[0], -1)
    re = I @ wc.T + Q @ ws.T
    im = Q @ wc.T - I @ ws.T
    aI, aQ, aws, awc = np.abs(I), np.abs(Q), np.abs(ws), np.abs(wc)
    return re, im, aI @ awc.T + aQ @ aws.T, aQ @ awc.T + aI @ aws.T


def epilogue_oracle(re, im, N, F, n_fft, shift=None):
    """(N, n_fft, F): ln(|X| + 1e-6), bin b at row (b + n/2) % n"""
    shift = n_fft // 2 if shift is None else shift
    mag = np.sqrt(np.asarray(re, np.float64) ** 2 + np.asarray(im, np.float64) ** 2)
    v = np.log(mag + 1e-6).reshape(N, F, n_fft).transpose(0, 2, 1)
    return np.roll(v, shift, axis=1)


def dc_oracle(re, im, gout, N, F, n_fft):
    """dL/dRe, dL/dIm (M, n_fft) from Re / Im and dL/d(out); 0 where |X| = 0 (the kernels' convention)"""
    re, im = np.asarray(re, np.float64), np.asarray(im, np.float64)
    g = np.roll(np.asarray(gout, np.float64), -(n_fft // 2), axis=1).transpose(0, 2, 1).reshape(N * F, n_fft)
    mag = np.sqrt(re * re + im * im)
    w = np.where(mag > 0, g / np.where(mag > 0, (mag + 1e-6) * mag, 1.0), 0.0)
    return w * re, w * im


def da_oracle(dre, dim, wsin, wcos):
    """dL/d(frame) (M, 2 n_fft) = [I part | Q part] and the abs-sums"""
    ws, wc = np.asarray(wsin, np.float64).reshape(wsin.shape[0], -1), np.asarray(wcos, np.float64).reshape(wcos.shape[0], -1)
    dre, dim = np.asarray(dre, np.float64), np.asarray(dim, np.float64)
    a, b, aws, awc = np.abs(dre), np.abs(dim), np.abs(ws), np.abs(wc)
    dA = np.concatenate([dre @ wc - dim @ ws, dre @ ws + dim @ wc], 1)
    S = np.concatenate([a @ awc + b @ aws, a @ aws + b @ awc], 1)
    return dA, S


def fold_oracle(dA, N, T, n_fft, hop, frames, skip_left_mirror=False):
    """dL/d(iq) (N, T, 2) from the frame gradients dA (N F', 2 n_fft) of the frames `frames` (F' indices): overlap-add into
    the padded positions, then each padded position u to the sample reflect(u) it holds.  Also sum|terms| and the number of
    terms per sample.  skip_left_mirror: a deliberately wrong variant that drops u < n_fft/2."""
    frames = np.asarray(frames, dtype=np.int64)
    Fp, Up = len(frames), T + n_fft
    d = np.asarray(dA, np.float64).reshape(N, Fp, 2, n_fft)
    G, A, cnt = np.zeros((N, 2, Up)), np.zeros((N, 2, Up)), np.zeros(Up)
    for i, f in enumerate(frames):
        sl = slice(f * hop, f * hop + n_fft)
        G[:, :, sl] += d[:, i]
        A[:, :, sl] += np.abs(d[:, i])
        cnt[sl] += 1
    u = np.arange(Up)
    if skip_left_mirror:
        u = u[u >= n_fft // 2]
    t = reflect(u, T, n_fft)
    g, a, c = np.zeros((T, N, 2)), np.zeros((T, N, 2)), np.zeros(T)
    np.add.at(g, t, G[:, :, u].transpose(2, 0, 1))
    np.add.at(a, t, A[:, :, u].transpose(2, 0, 1))
    np.add.at(c, t, cnt[u])
    return g.transpose(1, 0, 2), a.transpose(1, 0, 2), c


def kgrad_oracle(dre, dim, I, Q):
    """dL/dwsin, dL/dwcos (n_fft, n_fft) and the abs-sums"""
    dre, dim = np.asarray(dre, np.float64), np.asarray(dim, np.float64)
    a, b, aI, aQ = np.abs(dre), np.abs(dim), np.abs(I), np.abs(Q)
    return (dre.T @ Q - dim.T @ I, dre.T @ I + dim.T @ Q, a.T @ aQ + b.T @ aI, a.T @ aI + b.T @ aQ)


# ---- the criteria ---------------------------------------------------------------------------------------------------------
def gamma(K):
    """relative bound of one GEMM entry with K products (module docstring)"""
    K = 32 * -(-K // 32)
    return SAFETY * (2.0 ** -22 + 2.0 ** -20 + (K / 4) * 2.0 ** -23 + (K / 4) * 2.0 ** -33 + 3 * U24)


def gamma_dbt(kb_per_split, splits):
    return gamma(32 * kb_per_split) + SAFETY * splits * U24


def ratio(got, want, bound):
    """worst |got - want| / bound; an error where the bound is 0 (or a NaN) counts as infinite"""
    err = np.abs(np.asarray(got, np.float64) - want)
    err = np.where(np.isnan(err), np.inf, err)
    r = np.where(bound > 0, err / np.where(bound > 0, bound, 1.0), np.where(err > 0, np.inf, 0.0))
    return float(r.max()) if r.size else 0.0


def check_forward(re32, im32, I, Q, wsin, wcos):
    re, im, sre, sim = forward_oracle(I, Q, wsin, wcos)
    K = 2 * I.shape[1]
    return max(ratio(re32, re, gamma(K) * sre), ratio(im32, im, gamma(K) * sim))


def check_epilogue(out, re32, im32, N, F, n_fft):
    want = epilogue_oracle(re32, im32, N, F, n_fft)
    ulp = np.spacing(np.abs(want).astype(np.float32)).astype(np.float64)
    return ratio(out, want, 4 * ulp + 2.0 ** -22)


def check_dc(dre32, dim32, re32, im32, gout, N, F, n_fft):
    dre, dim = dc_oracle(re32, im32, gout, N, F, n_fft)
    return max(ratio(dre32, dre, 16 * U24 * np.abs(dre)), ratio(dim32, dim, 16 * U24 * np.abs(dim)))


def check_da(da32, dre32, dim32, wsin, wcos):
    dA, S = da_oracle(dre32, dim32, wsin, wcos)
    return ratio(da32, dA, gamma(da32.shape[1]) * S)


def check_fold(giq, da32, N, T, n_fft, hop, frames):
    g, a, c = fold_oracle(da32, N, T, n_fft, hop, frames)
    return ratio(giq, g, c[None, :, None] * U24 * a)


def check_kgrad(gsin, gcos, dre32, dim32, I, Q, kb_per_split, splits):
    gs, gc, ss, sc = kgrad_oracle(dre32, dim32, I, Q)
    gm = gamma_dbt(kb_per_split, splits)
    return max(ratio(gsin, gs, gm * ss), ratio(gcos, gc, gm * sc))


# ---- CPU: the oracle ------------------------------------------------------------------------------------------------------
def _kernels64(n_fft, seed, perturb=0.03):
    from skeleton_action_recognition_b200.layers.virtual_radar import _STFTKernels
    wsin, wcos = _STFTKernels.analytic(n_fft)
    g = np.random.default_rng(seed)
    wsin = (wsin.numpy() + perturb * g.standard_normal(wsin.shape)).astype(np.float32)
    wcos = (wcos.numpy() + perturb * g.standard_normal(wcos.shape)).astype(np.float32)
    return wsin, wcos


def _torch_kernels(wsin, wcos, hop):
    from skeleton_action_recognition_b200.layers.virtual_radar import _STFTKernels
    k = _STFTKernels(wsin.shape[0], hop, True, "cpu").double()
    with torch.no_grad():
        k.wsin.copy_(torch.from_numpy(wsin).double())
        k.wcos.copy_(torch.from_numpy(wcos).double())
    return k


@pytest.mark.parametrize("N,T,n_fft,hop", [(2, 9, 16, 3), (3, 77, 32, 5), (2, 300, 64, 16), (1, 129, 256, 40), (2, 40, 32, 50)])
def test_oracle_equals_the_torch_restatement_and_nnaudio(N, T, n_fft, hop):
    """forward + epilogue in float64 against _STFTKernels._logmag_torch and oracle/nnaudio_stft.py (both float64); the pad
    oracle against torch's reflect padding; the backward chain (dc, dA, fold, kernel gradients) against float64 autograd."""
    from oracle import virtual_radar_oracle as vro
    from oracle.nnaudio_stft import STFT
    rng = np.random.default_rng(T)
    iq = rng.standard_normal((N, T, 2)).astype(np.float32)
    wsin, wcos = _kernels64(n_fft, T)
    F = T // hop + 1
    Lp = (T + n_fft + 3) & ~3
    P = pad_oracle(iq, n_fft, Lp)
    zp = torch.nn.functional.pad(torch.from_numpy(iq).permute(0, 2, 1), (n_fft // 2, n_fft // 2), mode="reflect").numpy()
    assert np.array_equal(P[:, :, :T + n_fft], zp) and not P[:, :, T + n_fft:].any()
    I, Q = frame_rows(P, F, n_fft, hop)
    re, im, _, _ = forward_oracle(I, Q, wsin, wcos)
    out = epilogue_oracle(re, im, N, F, n_fft)
    k = _torch_kernels(wsin, wcos, hop)
    x = torch.from_numpy(iq).double().requires_grad_(True)
    ref = k._logmag_torch(x)
    np.testing.assert_allclose(out, ref.detach().numpy(), rtol=0, atol=1e-10)
    st = STFT(n_fft=n_fft, freq_bins=n_fft, hop_length=hop, output_format="Complex", device="cpu").double()
    st.wsin.data, st.wcos.data = torch.from_numpy(wsin).double(), torch.from_numpy(wcos).double()
    np.testing.assert_allclose(out, vro.stft_logmag(torch.from_numpy(iq).double(), st, n_fft).numpy(), rtol=0, atol=1e-10)
    # the backward chain, each stage fed the previous stage's float64 result
    gout = rng.standard_normal(out.shape)
    (ref * torch.from_numpy(gout)).sum().backward()
    dre, dim = dc_oracle(re, im, gout, N, F, n_fft)
    dA, _ = da_oracle(dre, dim, wsin, wcos)
    g, _, _ = fold_oracle(dA, N, T, n_fft, hop, np.arange(F))
    gs, gc, _, _ = kgrad_oracle(dre, dim, I, Q)
    for got, want in ((g, x.grad), (gs, k.wsin.grad[:, 0]), (gc, k.wcos.grad[:, 0])):
        want = want.numpy()
        np.testing.assert_allclose(got, want, rtol=0, atol=1e-10 * np.abs(want).max())


def test_oracle_kept_route_and_zero_magnitude():
    """The kept route's oracle (compact copy, fold over the kept frames) equals the full route's with the other frames'
    gradients zeroed; and at |X| = 0 (an all-zero sequence) float64 autograd gives NaN where the oracle -- like the
    kernels -- gives 0: a deliberate difference."""
    N, T, n_fft, hop = 2, 203, 32, 6
    F = T // hop + 1
    rng = np.random.default_rng(7)
    iq = rng.standard_normal((N, T, 2)).astype(np.float32)
    frames = np.array([0, 5, 6, 20, F - 1], dtype=np.int32)
    Pk = gather_oracle(iq, frames, n_fft, hop)
    Pf = pad_oracle(iq, n_fft, (T + n_fft + 3) & ~3)
    Ik, Qk = frame_rows(Pk, len(frames), n_fft, n_fft)
    If, Qf = frame_rows(Pf, F, n_fft, hop)
    rows = (np.arange(N)[:, None] * F + frames).ravel()
    assert np.array_equal(Ik, If[rows]) and np.array_equal(Qk, Qf[rows])
    dA = rng.standard_normal((N * len(frames), 2 * n_fft))
    full = np.zeros((N * F, 2 * n_fft))
    full[rows] = dA
    gk, _, ck = fold_oracle(dA, N, T, n_fft, hop, frames)
    gf, _, _ = fold_oracle(full, N, T, n_fft, hop, np.arange(F))
    np.testing.assert_allclose(gk, gf, rtol=0, atol=1e-12)
    assert (ck == 0).any() and not gk[:, ck == 0].any()             # samples no kept frame covers
    wsin, wcos = _kernels64(n_fft, 1)
    iq[0] = 0
    I, Q = frame_rows(pad_oracle(iq, n_fft, T + n_fft), F, n_fft, hop)
    re, im, _, _ = forward_oracle(I, Q, wsin, wcos)
    assert not re[:F].any() and not im[:F].any()
    dre, dim = dc_oracle(re, im, np.ones((N, n_fft, F)), N, F, n_fft)
    assert not dre[:F].any() and np.isfinite(dre).all()
    x = torch.from_numpy(iq).double().requires_grad_(True)
    _torch_kernels(wsin, wcos, hop)._logmag_torch(x).sum().backward()
    assert torch.isnan(x.grad[0]).all() and torch.isfinite(x.grad[1]).all()


# ---- CPU: the criteria have teeth ---------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def cabi():
    import __graft_entry__ as ge
    ge.build_product()
    from skeleton_action_recognition_b200 import _cabi
    return _cabi


def _synthetic(N, T, n_fft, hop, seed):
    """a float32 case built in numpy: every stage's 'kernel output' is the float64 oracle rounded to float32"""
    rng = np.random.default_rng(seed)
    iq = rng.standard_normal((N, T, 2)).astype(np.float32)
    wsin, wcos = _kernels64(n_fft, seed)
    F = T // hop + 1
    P = pad_oracle(iq, n_fft, (T + n_fft + 3) & ~3)
    I, Q = frame_rows(P, F, n_fft, hop)
    re, im, _, _ = forward_oracle(I, Q, wsin, wcos)
    re32, im32 = re.astype(np.float32), im.astype(np.float32)
    gout = rng.standard_normal((N, n_fft, F)).astype(np.float32)
    dre, dim = dc_oracle(re32, im32, gout, N, F, n_fft)
    dre32, dim32 = dre.astype(np.float32), dim.astype(np.float32)
    return dict(iq=iq, wsin=wsin, wcos=wcos, F=F, I=I, Q=Q, re32=re32, im32=im32, gout=gout, dre32=dre32, dim32=dim32)


@pytest.mark.parametrize("n_fft", [16, 64, 256])
def test_criteria_accept_the_rounded_oracle_and_reject_wrong_forward_variants(n_fft):
    N, hop = 3, 7
    T = 2 * n_fft + 5
    d = _synthetic(N, T, n_fft, hop, n_fft)
    F, I, Q, re32, im32 = d["F"], d["I"], d["Q"], d["re32"], d["im32"]
    ws, wc = d["wsin"], d["wcos"]
    assert check_forward(re32, im32, I, Q, ws, wc) <= 1
    out32 = epilogue_oracle(re32, im32, N, F, n_fft).astype(np.float32)
    assert check_epilogue(out32, re32, im32, N, F, n_fft) <= 1
    assert check_dc(d["dre32"], d["dim32"], re32, im32, d["gout"], N, F, n_fft) <= 1
    dA, _ = da_oracle(d["dre32"], d["dim32"], ws, wc)
    assert check_da(dA.astype(np.float32), d["dre32"], d["dim32"], ws, wc) <= 1
    # a row shifted by one frame
    assert check_forward(np.roll(re32, 1, 0), np.roll(im32, 1, 0), I, Q, ws, wc) > 1
    # Re and Im of one bin swapped
    sre, sim = re32.copy(), im32.copy()
    sre[:, 3], sim[:, 3] = im32[:, 3], re32[:, 3]
    assert check_forward(sre, sim, I, Q, ws, wc) > 1
    # the fftshift off by one
    bad = epilogue_oracle(re32, im32, N, F, n_fft, shift=n_fft // 2 + 1).astype(np.float32)
    assert check_epilogue(bad, re32, im32, N, F, n_fft) > 1
    # one 32-column K block (of the natural [I | Q] order) left out of the forward sum
    A = np.concatenate([I, Q], 1)
    kb = (2 * n_fft // 32) // 2
    A[:, 32 * kb:32 * kb + 32] = 0
    bre, bim, _, _ = forward_oracle(A[:, :n_fft], A[:, n_fft:], ws, wc)
    assert check_forward(bre.astype(np.float32), bim.astype(np.float32), I, Q, ws, wc) > 1


def test_criteria_reject_wrong_gradient_variants(cabi):
    N, T, n_fft, hop = 3, 340, 64, 4
    p = cabi.plan_stft_general(N, T, n_fft, hop, 0, SMS)
    assert p["splits"] >= 2                                          # a slice to leave out
    d = _synthetic(N, T, n_fft, hop, 11)
    F, I, Q, dre32, dim32 = d["F"], d["I"], d["Q"], d["dre32"], d["dim32"]
    kbs, sp = p["kb_per_split"], p["splits"]
    gs, gc, _, _ = kgrad_oracle(dre32, dim32, I, Q)
    assert check_kgrad(gs.astype(np.float32), gc.astype(np.float32), dre32, dim32, I, Q, kbs, sp) <= 1
    # one split slice's frames missing
    keep = np.ones(N * F, bool)
    keep[32 * kbs:64 * kbs] = False
    bs, bc, _, _ = kgrad_oracle(dre32[keep], dim32[keep], I[keep], Q[keep])
    assert check_kgrad(bs.astype(np.float32), bc.astype(np.float32), dre32, dim32, I, Q, kbs, sp) > 1
    # the last frame of every sequence missing (a wrong wrap of the frame-column view)
    keep = np.arange(N * F) % F != F - 1
    bs, bc, _, _ = kgrad_oracle(dre32[keep], dim32[keep], I[keep], Q[keep])
    assert check_kgrad(bs.astype(np.float32), bc.astype(np.float32), dre32, dim32, I, Q, kbs, sp) > 1
    # the fold: accepted rounded, rejected without the left mirror
    dA = da_oracle(dre32, dim32, d["wsin"], d["wcos"])[0].astype(np.float32)
    g = fold_oracle(dA, N, T, n_fft, hop, np.arange(F))[0]
    assert check_fold(g.astype(np.float32), dA, N, T, n_fft, hop, np.arange(F)) <= 1
    bad = fold_oracle(dA, N, T, n_fft, hop, np.arange(F), skip_left_mirror=True)[0]
    assert check_fold(bad.astype(np.float32), dA, N, T, n_fft, hop, np.arange(F)) > 1


# ---- CPU: the case table reaches every regime of the host plan ----------------------------------------------------------
def _regimes(cabi, sm_count):
    seen = set()
    for case in CASES:
        N, T, n, hop, kept, off, zero = case
        frames = kept_frames(case)
        Fk = 0 if frames is None else len(frames)
        p = cabi.plan_stft_general(N, T, n, hop, Fk, sm_count)
        F, M = p["F"], p["M"]
        kb_all = -(-M // 32)
        assert M == N * F and p["ldm"] == -(-M // 4) * 4 and p["nb"] == min(n, 64)
        assert p["row_tiles"] == -(-M // 128) and p["col_tiles"] == -(-2 * n // 128) and p["kblocks"] == 2 * n // 32
        assert (p["splits"] - 1) * p["kb_per_split"] + p["kb_last"] == kb_all and 1 <= p["kb_last"] <= p["kb_per_split"]
        if frames is None:
            assert p["Lp"] >= T + n and p["Lp"] % 4 == 0 and p["hop_view"] == hop and F == T // hop + 1
            seen |= {"F=1"} if F == 1 else set()
            seen |= {"hop>n_fft"} if hop > n else set()
            seen |= {"hop%4!=0"} if hop % 4 else set()
            seen |= {"T=n/2+1"} if T == n // 2 + 1 else set()
            seen |= {"Lp padded"} if p["Lp"] > T + n else set()
            seen |= {"frames_work+1 at hop%4=0"} if "frames" in off and hop % 4 == 0 else set()
        else:
            assert p["Lp"] == Fk * n and p["hop_view"] == n and F == Fk
            assert (np.diff(frames) > 0).all() and 0 <= frames[0] and frames[-1] <= T // hop
            if kept[0] == "resize":
                seen.add("kept: resize table")
            seen |= {"kept: single frame"} if Fk == 1 else set()
            seen |= {"kept: first and last"} if list(frames) == [0, T // hop] else set()
            seen |= {"kept: gaps > n/hop"} if Fk > 1 and np.diff(frames).max() > n // hop else set()
        seen.add("n_fft=%d" % n)
        seen |= {"M<128"} if M < 128 else {"M%%128=%d" % (M % 128)}
        seen |= {"M%4!=0"} if M % 4 else set()
        seen |= {"M%%32=%d" % (M % 32)}
        seen |= {"F=%d" % F}
        seen.add("splits=1" if p["splits"] == 1 else "splits>1")
        seen |= {"last slice shorter"} if p["kb_last"] < p["kb_per_split"] else set()
        for kb in (p["kb_per_split"], p["kb_last"]):
            seen.add("kb/slice=%d" % kb if kb <= 8 else ("kb/slice>=13" if kb >= 13 else "kb/slice 9..12"))
        seen.add("tiles=%d splits=%s" % (p["dbt_tiles"], p["splits"] if p["dbt_tiles"] > 4 else "any"))
        seen |= {"more CTAs than SMs"} if p["dbt_tiles"] * p["splits"] > sm_count else set()
        seen |= {"da_work+1"} if "da" in off else set()
        seen |= {"dbt_work+1 splits=1"} if "dbt" in off and p["splits"] == 1 else set()
        seen |= {"iq+8B"} if "iq" in off else set()
        seen |= {"grad_iq+8B"} if "giq" in off else set()
        seen |= {"|X|=0"} if zero else set()
    return seen


REGIMES = ({"n_fft=%d" % n for n in (16, 32, 64, 128, 256, 512, 1024)}
           | {"M<128", "M%128=0", "M%128=1", "M%128=127", "M%4!=0"}
           | {"F=1", "hop>n_fft", "hop%4!=0", "T=n/2+1", "Lp padded"}
           | {"splits=1", "splits>1", "last slice shorter", "kb/slice>=13"} | {"kb/slice=%d" % k for k in range(1, 9)}
           | {"M%32=1", "M%32=4", "M%32=31", "F=1", "F=2", "F=3", "F=5"}
           | {"tiles=1 splits=any", "tiles=4 splits=any", "tiles=16 splits=9", "tiles=64 splits=2", "tiles=256 splits=1",
              "more CTAs than SMs"}
           | {"kept: resize table", "kept: single frame", "kept: first and last", "kept: gaps > n/hop"}
           | {"frames_work+1 at hop%4=0", "da_work+1", "dbt_work+1 splits=1", "iq+8B", "grad_iq+8B", "|X|=0"})


def test_case_table_reaches_every_regime_of_the_plan(cabi):
    seen = _regimes(cabi, SMS)
    assert REGIMES <= seen, sorted(REGIMES - seen)
    # the feasibility examples of the table
    assert cabi.plan_stft_general(1, 2050, 256, 16)["M"] == 129
    assert cabi.plan_stft_general(3, 40, 32, 50)["F"] == 1
    p = cabi.plan_stft_general(1, 1600, 64, 1)
    assert (p["M"], p["splits"], p["kb_per_split"], p["kb_last"]) == (1601, 7, 8, 3)


# ---- GPU: every stage of every case --------------------------------------------------------------------------------------
def _run(case, sms):
    """Forward and backward through the C ABI with buffers the test owns (NaN-filled, so nothing unwritten passes) ->
    every intermediate, read back."""
    from skeleton_action_recognition_b200 import _cabi
    L = _cabi.lib()
    N, T, n, hop, kept, off, zero = case
    frames = kept_frames(case)
    Fk = 0 if frames is None else len(frames)
    p = _cabi.plan_stft_general(N, T, n, hop, Fk, sms)
    F, M, ldm = p["F"], p["M"], p["ldm"]
    parts = (ctypes.c_int64 * 3)()
    if frames is None:
        L.vr_stft_general_workspace_floats(N, T, n, hop, parts)
    else:
        L.vr_stft_general_frames_workspace_floats(N, Fk, n, parts)
    rng = np.random.default_rng(N * 7919 + T * 31 + n + hop)
    iq = rng.standard_normal((N, T, 2)).astype(np.float32)
    if zero:
        iq[0] = 0
    wsin, wcos = _kernels64(n, T + hop, perturb=0.02)
    gout = rng.standard_normal((N, n, F)).astype(np.float32)
    dev = torch.device("cuda:0")
    shift = {"frames": 1, "da": 1, "dbt": 1, "iq": 2, "giq": 2}       # floats: 4 or 8 bytes past 16-byte alignment
    bufs = {}

    def buf(name, floats, init=None):
        o = shift.get(name, 0) if name in off else 0
        t = torch.full((floats + o,), float("nan"), dtype=torch.float32, device=dev)
        if init is not None:
            t[o:] = torch.from_numpy(np.ascontiguousarray(init).ravel()).to(dev)
        bufs[name] = (t, o, floats)
        return t.data_ptr() + 4 * o

    def back(name):
        t, o, floats = bufs[name]
        return t[o:o + floats].cpu().numpy()

    q_iq = buf("iq", N * T * 2, iq)
    q_ws, q_wc = buf("wsin", n * n, wsin), buf("wcos", n * n, wcos)
    q_go = buf("gout", N * n * F, gout)
    q_fw, q_bt, q_cs = buf("frames", int(parts[0])), buf("bt", int(parts[1])), buf("csave", int(parts[2]))
    q_out, q_dc = buf("out", N * n * F), buf("dc", int(parts[2]))
    q_da, q_dbt, q_giq = buf("da", M * 2 * n), buf("dbt", int(parts[1])), buf("giq", N * T * 2)
    q_gs, q_gc = buf("gsin", n * n), buf("gcos", n * n)
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    if frames is None:
        rc = L.vr_stft_general_f32(q_iq, N, T, n, hop, q_ws, q_wc, q_fw, q_bt, q_cs, q_out, stream)
        _cabi.check(rc)
        rc = L.vr_stft_general_backward_f32(q_go, q_fw, q_bt, q_cs, N, T, n, hop, q_dc, q_da, q_dbt, q_giq, q_gs, q_gc, stream)
    else:
        tab = torch.from_numpy(frames).to(dev)
        rc = L.vr_stft_general_frames_f32(q_iq, N, T, n, hop, tab.data_ptr(), Fk, q_ws, q_wc, q_fw, q_bt, q_cs, q_out, stream)
        _cabi.check(rc)
        rc = L.vr_stft_general_frames_backward_f32(q_go, q_fw, q_bt, q_cs, N, T, n, hop, tab.data_ptr(), Fk, q_dc, q_da, q_dbt,
                                                   q_giq, q_gs, q_gc, stream)
    _cabi.check(rc)
    torch.cuda.synchronize()
    got = {k: back(k) for k in ("frames", "csave", "out", "dc", "da", "giq", "gsin", "gcos")}
    return p, frames, iq, wsin, wcos, gout, got


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_every_stage_against_the_float64_oracle(case):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    if sms != SMS:
        print("note: %d SMs, the case table was laid out for %d: the split-K regimes differ" % (sms, SMS))
    N, T, n, hop, kept, off, zero = case
    p, frames, iq, wsin, wcos, gout, got = _run(case, sms)
    F, M, ldm, Lp = p["F"], p["M"], p["ldm"], p["Lp"]
    rows = np.arange(F) if frames is None else frames
    # pad / gather: bit-equal
    P = got["frames"][:N * 2 * Lp].reshape(N, 2, Lp)
    want = pad_oracle(iq, n, Lp) if frames is None else gather_oracle(iq, frames, n, hop)
    assert np.array_equal(P.view(np.uint32), want.view(np.uint32)), "frames_work differs from the reflect padding"
    I, Q = frame_rows(P, F, n, p["hop_view"])
    re32, im32 = read_columns(got["csave"], n, ldm, M)
    dre32, dim32 = read_columns(got["dc"], n, ldm, M)
    dc_pad = got["dc"][:2 * n * ldm].reshape(2 * n, ldm)[:, M:]
    da32 = got["da"].reshape(M, 2 * n)
    giq = got["giq"].reshape(N, T, 2)
    r = {"forward": check_forward(re32, im32, I, Q, wsin, wcos),
         "epilogue": check_epilogue(got["out"].reshape(N, n, F), re32, im32, N, F, n),
         "dc": check_dc(dre32, dim32, re32, im32, gout, N, F, n),
         "dA": check_da(da32, dre32, dim32, wsin, wcos),
         "fold": check_fold(giq, da32, N, T, n, hop, rows),
         "dBt+dw": check_kgrad(got["gsin"].reshape(n, n), got["gcos"].reshape(n, n), dre32, dim32, I, Q,
                               p["kb_per_split"], p["splits"])}
    print("%s: worst err/bound %s" % (case_id(case), "  ".join("%s %.3g" % kv for kv in r.items())))
    assert not dc_pad.any() and np.isfinite(dc_pad).all(), "padding rows of dc_work are not 0"
    if zero:
        assert not re32[:F].any() and not dre32[:F].any() and not dim32[:F].any() and not giq[0].any()
    assert all(v <= 1 for v in r.values()), r
