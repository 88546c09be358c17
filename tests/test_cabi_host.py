"""CPU tests of the C-ABI library: it loads without a GPU, exports every symbol the header declares,
and its host-side logic (planner, bone partitioner, argument checks) behaves."""
import ctypes
import os
import re

import numpy as np
import pytest

from tests.conftest import ROOT


@pytest.fixture(scope="module")
def cabi():
    import __graft_entry__ as ge
    ge.build()
    from skeleton_action_recognition_b200 import _cabi
    return _cabi


def header_symbols():
    text = open(os.path.join(ROOT, "include", "virtual_radar_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(vr_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol(cabi):
    L = cabi.lib()
    names = header_symbols()
    assert set(names) == set(cabi.SYMBOLS), (names, cabi.SYMBOLS)
    for n in names:
        assert hasattr(L, n), n
    assert L.vr_abi_version() == 1


def test_plan_ntu(cabi):
    from skeleton_action_recognition_b200 import edges
    src, dst = map(list, zip(*edges))
    p = cabi.plan(256, 300, 25, 2, src, dst)
    assert p["frames_per_job"] == 19 and p["jobs_per_seq"] == 1 and p["grid"] == 256
    assert p["tma_loads"] == 1 and p["tma_bulk_store"] == 1
    assert p["chunks_per_job"] == 10 and p["chunk_steps"] == 32
    assert p["block"] == 288 and p["ring_stages"] >= 3
    assert p["smem_bytes"] <= 232448 // 2
    assert p["max_bones_per_group"] <= 7
    p = cabi.plan(65536, 300, 25, 2, src, dst)
    assert p["grid"] == 148 * p["ctas_per_sm"]
    p = cabi.plan(1, 165000, 25, 1, src, dst)
    assert p["jobs_per_seq"] * p["frames_per_job"] >= 10313 and p["tma_bulk_store"] == 0
    assert p["z_capacity"] >= (p["frames_per_job"] - 1) * 16 + 256
    p = cabi.plan(2, 301, 25, 1, src, dst)       # T*V*M not a multiple of 4 -> no TMA loads
    assert p["tma_loads"] == 0


def test_plan_team(cabi):
    """Team-job schedule (vr_team_kernel), host-only: two CTAs per SM, a two-stage ring per team whose stages can hold
    the output tile, picked automatically only for batches with several sequences per team slot."""
    from skeleton_action_recognition_b200 import edges
    src, dst = map(list, zip(*edges))
    p = cabi.plan_team(16384, 300, 25, 2, src, dst)
    assert p["grid"] == 296 and p["block"] == 320 and p["teams_per_cta"] == 2 and p["ring_stages_per_team"] == 2
    assert p["smem_bytes"] <= 233472 // 2 - 1024
    assert p["stage_bytes"] >= max(3 * 32 * 50 * 4, 256 * 19 * 4) and p["stage_bytes"] % 128 == 0
    assert p["z_stride"] >= 300 * 8 and p["automatic"] == 1
    assert cabi.plan_team(256, 300, 25, 2, src, dst)["automatic"] == 0
    assert cabi.plan_team(256, 300, 25, 2, src, dst)["grid"] == 128
    assert cabi.plan_team(7, 300, 25, 2, src, dst)["grid"] == 4
    assert cabi.plan_team(4, 300, 25, 1, src, dst)["grid"] == 2                # odd M: scalar twin
    for bad in ((4, 165000, 25, 1), (4, 301, 25, 1), (4, 400, 25, 2)):       # several jobs / no TMA loads / 26 frames: no single bulk store
        with pytest.raises(NotImplementedError):
            cabi.plan_team(*bad, src, dst)


def test_plan_image(cabi):
    """Launch plan of the fused resize (vr_forward_image_f32), host-only."""
    from skeleton_action_recognition_b200 import edges
    from oracle import resize
    src, dst = map(list, zip(*edges))
    p = cabi.plan_image(256, 300, 25, 2, src, dst, 256)
    assert p["columns"] == 256 and p["columns_per_job"] == 256 and p["jobs_per_seq"] == 1 and p["sparse_frames"] == 0
    assert p["frames_per_tile"] == 19 and p["tma_bulk_store"] == 0 and p["grid"] == 256
    p = cabi.plan_image(4, 75000, 25, 2, src, dst, 256)          # 4688 frames, 256 kept
    assert p["sparse_frames"] == 1 and p["columns"] == 256
    assert p["jobs_per_seq"] * p["columns_per_job"] >= 256
    # the widest job's samples fit the z buffer: (kept frames span) * hop + n_fft
    kept = resize.nearest_index(256, 4688)
    cj = p["columns_per_job"]
    span = max((kept[min(c0 + cj, 256) - 1] - kept[c0]) * 16 + 256 for c0 in range(0, 256, cj))
    assert span <= p["z_capacity"] <= 2304 + 16
    p = cabi.plan_image(2, 3000, 25, 2, src, dst, 256)           # 188 frames -> dense, several jobs
    assert p["sparse_frames"] == 0 and p["jobs_per_seq"] >= 2
    with pytest.raises(ValueError):
        cabi.plan_image(1, 300, 25, 2, src, dst, 5000)


def test_partition_keeps_sources_together_and_balances(cabi):
    from skeleton_action_recognition_b200 import edges
    src, dst = map(list, zip(*edges))
    grp = cabi.partition_edges(src, dst, 25)
    assert len(grp) == 24 and set(grp) <= {0, 1, 2, 3}
    by_src = {}
    for s, g in zip(src, grp):
        by_src.setdefault(s, set()).add(g)
    assert all(len(v) == 1 for v in by_src.values())
    counts = [grp.count(g) for g in range(4)]
    assert max(counts) <= 7 and min(counts) >= 5
    chain = [(i, i + 1) for i in range(41)]
    s2, d2 = map(list, zip(*chain))
    g2 = cabi.partition_edges(s2, d2, 42)
    assert sorted(g2.count(g) for g in range(4)) == [10, 10, 10, 11]
    star = [(0, i) for i in range(1, 9)]
    s3, d3 = map(list, zip(*star))
    assert len(set(cabi.partition_edges(s3, d3, 9))) == 1


def test_argument_errors(cabi):
    from skeleton_action_recognition_b200 import edges
    src, dst = map(list, zip(*edges))
    with pytest.raises(ValueError, match="exceed n_fft/2"):
        cabi.plan(1, 128, 25, 1, src, dst)
    cabi.plan(1, 129, 25, 1, src, dst)
    with pytest.raises(ValueError, match="outside"):
        cabi.plan(1, 300, 24, 1, src, dst)          # joint 24 does not exist
    with pytest.raises(NotImplementedError, match="n_fft=256"):
        cabi.plan(1, 300, 25, 1, src, dst, n_fft=512)
    with pytest.raises(ValueError):
        cabi.plan(0, 300, 25, 1, src, dst)
    with pytest.raises(ValueError):
        cabi.plan(1, 300, 25, 1, src, dst, hop=0)


def test_stft_general_rejects_misaligned_work_buffers(cabi):
    """Argument validation happens before any CUDA call: fake device addresses are enough (no GPU needed)."""
    L = cabi.lib()
    ok = 0x10000                                     # 16-byte aligned, never dereferenced: the call stops at the checks
    args = lambda bt, cs, iq=ok: (iq, 2, 300, 256, 16, ok, ok, ok, bt, cs, ok, None)      # noqa: E731
    assert L.vr_stft_general_f32(*args(ok + 4, ok)) == cabi.VR_ERR_ARG
    assert "16-byte" in cabi.last_error()
    assert L.vr_stft_general_f32(*args(ok, ok + 8)) == cabi.VR_ERR_ARG
    assert L.vr_stft_general_f32(*args(ok, None, ok + 4)) == cabi.VR_ERR_ARG
    assert L.vr_stft_general_f32(*args(None, ok)) == cabi.VR_ERR_ARG           # null work buffer
    # backward: dc_work misaligned
    assert L.vr_stft_general_backward_f32(ok, ok, ok, ok, 2, 300, 256, 16, ok + 4, None, None, None, None, None, None) == cabi.VR_ERR_ARG


def test_plan_stft_general(cabi):
    """Host plan of the general-kernel STFT's GEMMs (vr_plan_stft_general): what the launches reject, and the split-K
    kernel gradient's limits -- splits x tiles within one wave of min(SMs, 160) CTAs whenever it splits, and the slices'
    K x K planes within one slot of the static pool (160 tiles of 128 x 128 floats)."""
    L = cabi.lib()
    assert L.vr_plan_stft_general(2, 300, 256, 16, 0, 148, None) == cabi.VR_ERR_ARG
    for bad, exc in (((0, 300, 256, 16), ValueError), ((2, 300, 256, 0), ValueError), ((2, 128, 256, 16), ValueError),
                     ((2, 300, 48, 16), NotImplementedError), ((2, 300, 8, 16), NotImplementedError),
                     ((2, 3000, 2048, 16), NotImplementedError), ((1 << 27, 300, 256, 16), NotImplementedError)):
        with pytest.raises(exc):
            cabi.plan_stft_general(*bad)
    with pytest.raises(ValueError, match="F_kept"):
        cabi.plan_stft_general(2, 300, 256, 16, 20)                  # T / hop + 1 = 19 frames
    with pytest.raises(ValueError, match="F_kept"):
        cabi.plan_stft_general(2, 300, 256, 16, -1)
    assert cabi.plan_stft_general(2, 300, 256, 16, 19)["F"] == 19
    assert cabi.plan_stft_general(2, 300, 256, 16, 0, sm_count=0) == cabi.plan_stft_general(2, 300, 256, 16, 0, sm_count=148)
    p = cabi.plan_stft_general(4096, 300, 256, 16)                   # the flagship batch with trainable kernels
    assert (p["nb"], p["F"], p["M"], p["ldm"], p["Lp"]) == (64, 19, 77824, 77824, 556)
    assert (p["row_tiles"], p["col_tiles"], p["kblocks"], p["dbt_tiles"], p["splits"]) == (608, 4, 16, 16, 9)
    slot = 160 * 128 * 128
    for n in (16, 32, 64, 128, 256, 512, 1024):
        for N, T, hop in ((1, n // 2 + 1, 1), (3, 1000, 7), (64, 3000, 4), (4096, 300, 16), (20000, 2 * n, 1)):
            T = max(T, n // 2 + 1)
            for sms in (1, 16, 132, 148, 160, 1000):
                p = cabi.plan_stft_general(N, T, n, hop, 0, sms)
                K = 2 * n
                assert p["dbt_tiles"] == (-(-K // 128)) ** 2 and p["kblocks"] == K // 32 and p["col_tiles"] == -(-K // 128)
                kb_all = -(-p["M"] // 32)
                assert (p["splits"] - 1) * p["kb_per_split"] + p["kb_last"] == kb_all
                assert 1 <= p["kb_last"] <= p["kb_per_split"]
                if p["splits"] > 1:
                    assert p["splits"] * p["dbt_tiles"] <= min(sms, 160), (n, N, T, hop, sms, p)
                    assert p["splits"] * K * K <= slot, (n, N, T, hop, sms, p)


def test_module_surface_matches_reference():
    import torch
    from skeleton_action_recognition_b200 import VirtualRadar, edges
    assert len(edges) == 24 and edges[0] == (0, 1) and edges[-1] == (18, 19)
    layer = VirtualRadar(wavelength=5e-4, device="cpu")
    sd = layer.state_dict()
    assert list(sd.keys()) == ["wavelength", "radar_location", "stft.wsin", "stft.wcos"]
    assert sd["wavelength"].shape == () and sd["radar_location"].shape == (3,)
    assert sd["stft.wsin"].shape == (256, 1, 256) and sd["stft.wcos"].shape == (256, 1, 256)
    assert layer.src[:3] == [0, 1, 20] and layer.dst[:3] == [1, 20, 2] and layer.n_fft == 256
    assert not any(p.requires_grad for p in layer.parameters())
    # the STFT kernel parameters equal the oracle's nnAudio restatement bit for bit
    from oracle.nnaudio_stft import fourier_kernels
    wsin, wcos = fourier_kernels(256, 256)
    assert torch.equal(sd["stft.wsin"], torch.from_numpy(wsin))
    assert torch.equal(sd["stft.wcos"], torch.from_numpy(wcos))
    layer.stft.assert_dft()
    with pytest.raises(RuntimeError, match="no CPU path"):
        layer(torch.zeros(1, 3, 300, 25, 2))
    with pytest.raises(ValueError):
        layer(torch.zeros(1, 2, 300, 25, 2))
    trainable = VirtualRadar(train_wavelength=True, train_radar_location=True, device="cpu")   # reference flags, :40-42
    assert trainable.wavelength.requires_grad and trainable.radar_location.requires_grad
    assert not trainable.stft.wsin.requires_grad and not trainable._general_stft()
    tk = VirtualRadar(train_stft_kernel=True, device="cpu")
    assert tk.stft.wsin.requires_grad and tk.stft.wcos.requires_grad and not tk.wavelength.requires_grad
    assert tk._general_stft()                      # trainable kernels: synthesis kernel + GEMM STFT
    with torch.no_grad():
        assert tk._general_stft()                  # ... also for an eval pass: the optimizer may have moved the kernels
    # in-place edits through the parameters are seen (version counters), without a load_state_dict in between
    ed = VirtualRadar(device="cpu")
    assert not ed._general_stft()
    with torch.no_grad():
        ed.stft.wcos.mul_(1.5)
    assert ed._general_stft()
    with torch.no_grad():
        ed.stft.wcos.copy_(layer.stft.wcos)
    assert not ed._general_stft()
    import copy, pickle
    c = copy.deepcopy(layer)
    assert c.src == layer.src
    pickle.loads(pickle.dumps(layer))
    # reference-style checkpoints load
    layer2 = VirtualRadar(wavelength=1e-3, device="cpu")
    layer2.load_state_dict(sd)
    assert float(layer2.wavelength) == float(layer.wavelength)
    # ... but a checkpoint with TRAINED STFT kernels must not be silently replaced by the analytic DFT
    bad = {k: v.clone() for k, v in sd.items()}
    bad["stft.wsin"][3, 0, 5] += 0.25
    layer2.load_state_dict(bad)
    assert layer2._general_stft()                  # -> CUDA synthesis + GEMM against the loaded kernels
    with pytest.raises(NotImplementedError, match="analytic Hann-windowed DFT only"):
        layer2.forward_host(torch.zeros(1, 3, 300, 25, 2))
    layer2.load_state_dict(sd)
    assert not layer2._general_stft()
    with pytest.raises(RuntimeError, match="no CPU path"):
        layer2(torch.zeros(1, 3, 300, 25, 2))
    # the GEMM form of the STFT equals the oracle's nnAudio restatement (CPU, float32)
    from oracle import virtual_radar_oracle as vro
    from oracle.nnaudio_stft import STFT
    g = torch.Generator().manual_seed(4)
    iq = torch.randn(3, 400, 2, generator=g)
    ref = vro.stft_logmag(iq, STFT(n_fft=256, freq_bins=256, hop_length=16, device="cpu"), 256)
    got = layer2.stft._logmag_torch(iq)          # the torch restatement kept as a cross-check of the tcgen05 path (GPU tests)
    assert got.shape == ref.shape and torch.allclose(got, ref, atol=2e-4, rtol=0)


@pytest.mark.parametrize("T,hop,image", [(300, 16, 0), (300, 16, 256), (129, 16, 0), (5000, 16, 0), (75000, 16, 256),
                                         (75000, 16, 0), (4095, 16, 256), (4096, 16, 256), (20000, 16, 100), (9000, 16, 300),
                                         (3000, 16, 64), (700, 8, 256), (1001, 100, 128), (2500, 32, 77), (300, 16, 1),
                                         (165000, 16, 256), (6400, 16, 37), (333, 7, 19)])
def test_job_split_covers_every_column_and_fits_the_z_buffer(cabi, T, hop, image):
    """The job split (shared host/device code: col_frame, job_geom, the planner's column-per-job search): the jobs of a
    sequence tile its output columns exactly once, every frame a column shows has all of its reflect-padded samples
    inside the job's [lo, hi], and the span fits the planned z buffer and chunk count."""
    from oracle import resize
    from skeleton_action_recognition_b200 import edges
    src, dst = map(list, zip(*edges))
    F = T // hop + 1
    plan = cabi.plan_image(2, T, 25, 2, src, dst, image, hop=hop) if image else cabi.plan(2, T, 25, 2, src, dst, hop=hop)
    ncols = image if image else F
    fmap = resize.nearest_index(image, F) if image else np.arange(F)
    jps = plan["jobs_per_seq"]
    nxt = 0
    for j in range(jps):
        g = cabi.job_geometry(2, T, 25, 2, src, dst, jps + j, image_size=image, hop=hop)      # jobs of the second sequence
        assert g["sequence"] == 1 and g["first_column"] == nxt and g["columns"] >= 1
        nxt += g["columns"]
        cols = np.arange(g["first_column"], g["first_column"] + g["columns"])
        frames = fmap[cols]
        assert frames[0] == g["first_frame"] and frames[-1] == g["first_frame"] + g["frames"] - 1
        s = frames[:, None] * hop - 128 + np.arange(256)[None, :]
        s = np.abs(s)
        s = np.where(s >= T, 2 * (T - 1) - s, s)
        assert s.min() >= g["lo"] and s.max() <= g["hi"] and g["lo"] % 32 == 0 and 0 <= g["lo"] and g["hi"] <= T - 1
        assert g["hi"] - g["lo"] + 1 <= plan["z_capacity"] and g["chunks"] <= plan["chunks_per_job"]
        assert g["chunks"] == (g["hi"] - g["lo"]) // 32 + 1
    assert nxt == ncols
