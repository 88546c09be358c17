#!/usr/bin/env python
"""bench.py -- spectrograms/s of the VirtualRadar forward pass (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the hot path over one batch of BASELINE config 2
(N=256 NTU-shaped sequences, 3x300x25x2 -> 256x19) per GPU, synthetic input.

The K-step figures (value, stream_ordered, module_forward) are measured the same way (`timed_steps`): one untimed step
that loads the kernels, then at least W untimed steps, and at least 50 ms of them so that the clocks have risen, then
exactly K steps between two CUDA events on the launching stream, max over ranks.  The figures with a fixed size of
their own (large_batch, sweep) repeat their loop until at least 50 ms have been timed and report the median
repetition (`timed_reps`).

--dump-outputs DIR writes the spectrograms of the last timed step, (256, 256, 19) float32, to DIR/spectrograms.npy
(DIR/spectrograms_rank<r>.npy per rank on several GPUs).  The inputs are seeded, so two builds run with the same
arguments can be compared output for output.

  value          sequences/s, whole job, inputs resident in HBM, one fused launch per step, steps = independent batches
                 in distinct buffers (a pool larger than the 126 MB L2) launched with VR_FLAG_INPUTS_READY, so that
                 consecutive launches overlap (reads of step k+1 may start while step k's last CTAs finish; writes wait).
  stream_ordered the same loop in plain stream order -- what `VirtualRadar.forward` does by default.
  module_forward the drop-in module itself (`layer(x)`: checks, torch.empty, ctypes, launch), eager and as a CUDA graph.
  e2e            the same metric through the public API with HOST buffers: VirtualRadar.forward_host
                 (C ABI vr_forward_host_f32): pinned host input -> H2D -> kernel -> D2H inside the timed region.
  roofline       HBM bound: algorithmic bytes per launch (199456 B/spectrogram x 256, DESIGN.md) over the mean launch
                 duration measured here; peak from MEASURED_PEAKS.json (else the profiling guide's fallback).
  large_batch    one launch over 16384 sequences per GPU (the sustained figure).
  sweep          BASELINE config 4: global batches of 1k..64k sequences SHARDED by sequence over the ranks
                 (shard_bounds = DataParallel's split, main_spectrogram.py:118-119): aggregate rate per global N.
  shard_verify   (N > 1) a sharded batch, all-gathered over NCCL, is bit-identical to rank 0's single-GPU result.
  e2e_upsampled  the loader's pipeline end to end: raw pinned host batch -> H2D -> fused up-sampling x250 + radar + resize.
  train_step     BASELINE config 5 (1 GPU): main_spectrogram.py:146-158's step -- Model = fused radar input stage +
                 ResNet-18 (reference layout), batch 64, forward + backward + Adam -- with the input stage's share.
  cpu_baseline   the oracle port (reference algorithm, CPU PyTorch, all host threads) on this box's host cores.
  --impl reference   times only that CPU port, in the same JSON shape.
"""
import argparse
import hashlib
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the benchmark writes nothing into the tree it runs from (it may be read-only)

BATCH, T, V, M = 256, 300, 25, 2
N_FFT, HOP = 256, 16
F = T // HOP + 1
BYTES_IN = 4 * 3 * T * V * M                      # 180 000
BYTES_OUT = 4 * N_FFT * F                         # 19 456
BYTES_PER_SPEC = BYTES_IN + BYTES_OUT             # 199 456  (SURVEY 8d)
FLOPS_PER_SPEC = 55 * T * 24 * M + F * (5 * N_FFT * 8 + 8 * N_FFT)   # 1 025 472 (SURVEY 8d)
WAVELENGTH = 5e-4
WORKLOAD = "synthetic NTU-60 batch N=256, C=3, T=300, V=25, M=2 (BASELINE configs[1]), wavelength 5e-4, default 24-bone skeleton"
MIN_TIMED_MS = 50.0
MIN_WARM_MS = 50.0


def synth_batch(n, seed):
    """S1 of SURVEY 8d: seeded iid randn * 0.3 (CPU generator)."""
    import torch
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n, 3, T, V, M, generator=g) * 0.3


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def source_hash():
    """Hash of the kernel sources + header: ties a committed ncu capture to the build it was taken on."""
    h = hashlib.sha256()
    base = os.path.join(ROOT, "skeleton_action_recognition_b200", "csrc")
    for name in sorted(os.listdir(base)):
        with open(os.path.join(base, name), "rb") as f:
            h.update(name.encode() + b"\0" + f.read())
    with open(os.path.join(ROOT, "include", "virtual_radar_b200.h"), "rb") as f:
        h.update(f.read())
    return h.hexdigest()[:16]


def ncu_traffic(kernel_key):
    """dram bytes per launch from the committed `ncu --set full` capture (profiles/traffic.json, written by
    tools/ncu_summary.py) -- only if it was taken on THIS build of the kernels; otherwise null and the reason."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)
    except Exception:
        return None, "no committed capture"
    if t.get("source_hash") != source_hash():
        return None, "committed capture is of build %s, this is %s" % (t.get("source_hash"), source_hash())
    return t.get(kernel_key), t.get("source")


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU with NVML while the timed regions run."""

    def __init__(self, index, period=0.02):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.active = threading.Event()

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                     nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
                     nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake"}
            while not self._stop_evt.is_set():
                if self.active.is_set():
                    self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    for bit, name in names.items():
                        if r & bit:
                            self.reasons.add(name)
                time.sleep(self.period)
        except Exception as e:  # NVML missing: report nothing rather than fail the bench
            self.reasons.add("nvml_unavailable:%s" % type(e).__name__)

    def stop(self):
        self._stop_evt.set()

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


def physical_gpu_index(local):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local])
        except Exception:
            return local
    return local


# ----------------------------------------------------------------------------------------------
# CPU reference arm (oracle port == the reference's algorithm on CPU PyTorch)
# ----------------------------------------------------------------------------------------------
def time_cpu_port(n_seq, repeats, warmup=0):
    import torch
    from oracle import virtual_radar_oracle as vro
    torch.set_num_threads(os.cpu_count())
    o = vro.OracleVirtualRadar(wavelength=WAVELENGTH)
    x = synth_batch(n_seq, 0)
    for _ in range(warmup):
        o(x)
    times = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        o(x)
        times.append(time.perf_counter() - t0)
    return times


def run_reference(args, rank, world):
    """--impl reference: only rank 0 works; each step is a bounded sample of the workload sized so
    that warmup+steps finish in about two minutes (the CPU path does ~70-140 spectrograms/s)."""
    if rank != 0:
        return
    import torch
    total = args.steps + args.warmup
    n_seq = int(max(1, min(BATCH, (120.0 * 72.0) // max(1, total))))
    times = time_cpu_port(n_seq, args.steps, warmup=args.warmup)
    elapsed = sum(times)
    value = n_seq * args.steps / elapsed
    cores = torch.get_num_threads()
    sample = "%d of the %d sequences of the batch per step, %d steps" % (n_seq, BATCH, args.steps)
    line = {"impl": "reference", "metric": "spectrograms/sec (NTU 3x300x25x2)", "value": value,
            "unit": "spectrograms/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * elapsed / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "batch_per_gpu": BATCH, "sample_per_step": n_seq,
                       "note": "reference algorithm on CPU PyTorch (oracle port of layers/virtual_radar.py + nnAudio STFT restatement); rank 0 only"},
            "cpu_baseline": {"value": value, "unit": "spectrograms/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "spectrograms/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------
def run_ours(args, rank, world, local_rank):
    import ctypes
    import torch
    import numpy as np
    import torch.distributed as dist
    # the library __graft_entry__.build() left in the tree; nothing is compiled here (_cabi fails loudly if it is missing)
    from skeleton_action_recognition_b200 import VirtualRadar, _cabi, shard_bounds
    assert _cabi.lib().vr_abi_version() == _cabi.ABI_VERSION

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(values):
        if world == 1:
            return list(values)
        t = torch.tensor(list(values), dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]

    stream = torch.cuda.current_stream(dev)

    def timed_steps(step, k):
        """(milliseconds of exactly k steps, max over ranks; number of warm-up steps).  Warm-up: one step and a
        synchronize (a kernel's first launch loads its module, which must not count as warm-up time), then steps until
        at least args.warmup of them have been launched over at least MIN_WARM_MS.  The window then opens behind them
        without a synchronize, so the first timed step does not wait for its launch.  Warm-up steps have indices
        counting from 0, the timed steps 0..k-1: what the timed steps compute does not depend on the warm-up."""
        barrier()
        step(0)
        barrier()
        n, t0 = 1, time.perf_counter()
        while n < args.warmup or (time.perf_counter() - t0) * 1e3 < MIN_WARM_MS:
            step(n)
            n += 1
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(k):
            step(i)
        e1.record(stream)
        barrier()
        return max_over_ranks([e0.elapsed_time(e1)])[0], n

    def timed_reps(step, k, min_ms=MIN_TIMED_MS, max_reps=400, warm=3):
        """Median (over repetitions, after max over ranks) milliseconds of a k-step loop; repetitions until >= min_ms
        have been timed.  Each repetition is bracketed by barrier + synchronize; CUDA events on the launching stream."""
        for i in range(warm):
            step(i)
        barrier()
        reps, total, times = 0, 0.0, []
        while reps < 3 or (total < min_ms and reps < max_reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            e0.record(stream)
            for i in range(k):
                step(i)
            e1.record(stream)
            barrier()
            ms = e0.elapsed_time(e1)
            if world > 1:   # every rank must take the same number of repetitions: decide on the slowest rank's clock
                ms = max_over_ranks([ms])[0]
            times.append(ms)
            total += ms
            reps += 1
        times.sort()
        return times[len(times) // 2], reps, total

    layer = VirtualRadar(wavelength=WAVELENGTH, device=dev).to(dev)
    # pool of distinct batches bigger than L2 (126 MB): 6 x (46.1 + 5.0) MB = 306 MB
    pool = 6
    xs = [synth_batch(BATCH, 1000 * rank + i).to(dev) for i in range(pool)]
    outs = [torch.empty(BATCH, N_FFT, F, device=dev) for _ in range(pool)]
    lib = _cabi.lib()
    s_ptr = ctypes.c_void_p(stream.cuda_stream)
    lam_ptr, loc_ptr = layer.wavelength.data_ptr(), layer.radar_location.data_ptr()
    E = len(layer.src)
    K = args.steps

    def raw_step(i, flags):
        # the module's forward minus torch.empty: the same C-ABI call on preallocated buffers
        rc = lib.vr_forward_f32(xs[i % pool].data_ptr(), BATCH, T, V, M, layer._src_c, layer._dst_c, E,
                                lam_ptr, loc_ptr, N_FFT, HOP, flags, outs[i % pool].data_ptr(), s_ptr)
        if rc:
            _cabi.check(rc)

    sampler = ClockSampler(physical_gpu_index(local_rank))
    sampler.start()
    peak, peak_src = measured_peaks()
    frac = lambda n, ms: BYTES_PER_SPEC * n / (ms * 1e-3) / 1e9 / peak     # noqa: E731

    # ---- headline: device-resident throughput, independent batches ----------------------------
    sampler.active.set()
    ms_k, warm_n = timed_steps(lambda i: raw_step(i, _cabi.VR_FLAG_INPUTS_READY), K)
    sampler.active.clear()
    ms_per_step = ms_k / K
    value = world * BATCH / (ms_per_step * 1e-3)
    # correctness guard: the timed launches produced the same bits as the module's forward
    torch.cuda.synchronize(dev)
    for i in {0, (K - 1) % pool, K % pool}:
        assert torch.equal(outs[i], layer(xs[i])), "timed path != VirtualRadar.forward"
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        name = "spectrograms.npy" if world == 1 else "spectrograms_rank%d.npy" % rank
        np.save(os.path.join(args.dump_outputs, name), outs[(K - 1) % pool].cpu().numpy())

    # ---- the same loop in plain stream order (what the module does by default) ----------------
    sampler.active.set()
    so_k, so_warm = timed_steps(lambda i: raw_step(i, 0), K)
    so_ms = so_k / K
    # ---- the drop-in module itself: eager, and one forward captured in a CUDA graph ------------
    holder = [None]

    def module_step(i):
        holder[0] = layer(xs[i % pool])
    me_k, _ = timed_steps(module_step, K)
    me_ms = me_k / K
    static_x = xs[0].clone()
    side = torch.cuda.Stream(dev)
    side.wait_stream(stream)
    with torch.cuda.stream(side):
        layer(static_x)
    stream.wait_stream(side)
    torch.cuda.synchronize(dev)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static_y = layer(static_x)
    mg_k, _ = timed_steps(lambda i: graph.replay(), K)
    mg_ms = mg_k / K
    assert torch.equal(static_y, layer(static_x))
    sampler.active.clear()
    module_forward = {
        "eager": {"value": world * BATCH / (me_ms * 1e-3), "ms_per_step": me_ms, "hbm_frac": frac(BATCH, me_ms),
                  "note": "layer(x) per step on the device-resident pool: input checks, torch.empty, ctypes call, one launch, plain stream order"},
        "cuda_graph": {"value": world * BATCH / (mg_ms * 1e-3), "ms_per_step": mg_ms, "hbm_frac": frac(BATCH, mg_ms),
                       "note": "one layer(x) captured with torch.cuda.graph and replayed (same buffers every step, so the batch stays in L2)"}}
    del graph, static_x, static_y

    # ---- end to end through the public API with host buffers --------------------------------
    xh = [synth_batch(BATCH, 2000 * rank + i).pin_memory() for i in range(2)]
    oh = torch.empty(BATCH, N_FFT, F).pin_memory()
    e2e_steps = max(3, min(K, 200))
    while e2e_steps * 1.0 < MIN_TIMED_MS and e2e_steps < 200:      # ~1 ms per step: at least 50 ms
        e2e_steps *= 2
    for i in range(3):
        layer.forward_host(xh[i % 2], out=oh)
    barrier()
    sampler.active.set()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        layer.forward_host(xh[i % 2], out=oh)
    torch.cuda.synchronize(dev)
    dt = time.perf_counter() - t0
    sampler.active.clear()
    dt = max_over_ranks([dt])[0]
    e2e_value = world * BATCH * e2e_steps / dt
    assert torch.equal(oh, layer(xh[(e2e_steps - 1) % 2].to(dev)).cpu()), "e2e path != VirtualRadar.forward"
    del xh, oh

    # ---- sustained large batch (many jobs per team), for the roofline picture ----------------
    big_n = 16384
    base = synth_batch(256, 77 + rank).to(dev)
    xb = base.repeat(big_n // 256, 1, 1, 1, 1)
    ob = torch.empty(big_n, N_FFT, F, device=dev)

    def big_step(i):
        rc = lib.vr_forward_f32(xb.data_ptr(), big_n, T, V, M, layer._src_c, layer._dst_c, E, lam_ptr, loc_ptr,
                                N_FFT, HOP, 0, ob.data_ptr(), s_ptr)
        if rc:
            _cabi.check(rc)
    sampler.active.set()
    big_k, _, _ = timed_reps(big_step, 10, min_ms=100.0)
    sampler.active.clear()
    big_ms = big_k / 10
    big_value = world * big_n / (big_ms * 1e-3)
    del ob

    # ---- BASELINE config 4: global batches sharded by sequence over the ranks -----------------
    sweep = []
    for gn in (1024, 4096, 16384, 65536):
        lo, hi = shard_bounds(gn, world, rank)
        n_loc = hi - lo
        xsw = xb[:n_loc] if n_loc <= big_n else base.repeat((n_loc + 255) // 256, 1, 1, 1, 1)[:n_loc]
        osw = torch.empty(max(n_loc, 1), N_FFT, F, device=dev)

        def sw_step(i):
            if n_loc > 0:
                rc = lib.vr_forward_f32(xsw.data_ptr(), n_loc, T, V, M, layer._src_c, layer._dst_c, E, lam_ptr, loc_ptr,
                                        N_FFT, HOP, 0, osw.data_ptr(), s_ptr)
                if rc:
                    _cabi.check(rc)
        ksw = 8 if gn <= 4096 else 3
        sw_k, _, _ = timed_reps(sw_step, ksw, min_ms=30.0)
        sw_ms = sw_k / ksw
        sweep.append({"global_n": gn, "per_rank": -(-gn // world), "ms": sw_ms, "value": gn / (sw_ms * 1e-3),
                      "hbm_frac_per_gpu": frac(gn, sw_ms) / world})
        del osw, xsw
    # ---- shard verification: NCCL gathers the shards' outputs; nothing else crosses GPUs --------
    shard_verify = None
    if world > 1:
        from skeleton_action_recognition_b200 import sharded_forward
        vn = 1000                                      # not a multiple of the world size: ragged last shard
        xv = synth_batch(256, 4242).to(dev).repeat(4, 1, 1, 1, 1)[:vn].contiguous()
        xv[500:] *= 1.5
        full = sharded_forward(layer, xv)
        same = bool(torch.equal(full, layer(xv)))
        flag = torch.tensor([1.0 if same else 0.0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        shard_verify = {"global_n": vn, "world": world, "bit_identical_to_single_gpu": bool(flag.item() == 1.0),
                        "how": "shard_bounds split, each rank's fused launch, torch.distributed.all_gather_into_tensor (NCCL), torch.equal against the rank's own single-GPU result of the whole batch"}
        assert shard_verify["bit_identical_to_single_gpu"], "sharded result differs from single GPU"
        del xv, full
    sampler.stop()

    achieved = BYTES_PER_SPEC * BATCH / (ms_per_step * 1e-3) / 1e9
    big_achieved = BYTES_PER_SPEC * big_n / (big_ms * 1e-3) / 1e9
    props = torch.cuda.get_device_properties(dev)
    fp32_peak = props.multi_processor_count * 128 * 2 * 1.965e9 / 1e12
    plan = _cabi.plan(BATCH, T, V, M, layer.src, layer.dst, N_FFT, HOP, props.multi_processor_count)
    plan_team = _cabi.plan_team(BATCH, T, V, M, layer.src, layer.dst, N_FFT, HOP, props.multi_processor_count)

    def timed(fn, reps):
        for _ in range(2):
            fn()
        torch.cuda.synchronize(dev)
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record(stream)
        for _ in range(reps):
            fn()
        t1.record(stream)
        torch.cuda.synchronize(dev)
        return t0.elapsed_time(t1) / reps

    # ---- end to end for the loader's real pipeline: RAW pinned host batch -> H2D -> up-sampling x250 + radar + resize in
    # one fused pass -> image left on the device for the classifier (wall clock, copies inside the timed region, all
    # ranks at once, max over ranks).  PCIe carries 180 kB per sequence instead of the reference's 45 MB.
    un, uk, S = 2 * props.multi_processor_count, 250, 256
    uh = [synth_batch(un, 56 + i + 10 * rank).pin_memory() for i in range(2)]

    def from_host(i):
        return layer.forward_upsampled(uh[i % 2].to(dev, non_blocking=True), uk, 3, image_size=S)
    for i in range(2):
        from_host(i)
    barrier()
    t0 = time.perf_counter()
    for i in range(8):
        img = from_host(i)
    torch.cuda.synchronize(dev)
    dt = max_over_ranks([(time.perf_counter() - t0) / 8])[0]
    e2e_upsampled = {"value": world * un / dt, "unit": "sequences/s", "h2d_bytes_per_step": un * BYTES_IN, "d2h_bytes_per_step": 0,
                     "sequences_per_step_per_gpu": un, "frames_per_sequence": T * uk,
                     "api": "VirtualRadar.forward_upsampled(x.to(device), 250, 3, image_size=256) on a pinned raw batch",
                     "note": "raw (N,3,300,25,2) pinned host batch in, (N,1,256,256) image left on the device for the classifier; "
                             "the reference ships the 250x up-sampled batch (45 MB per sequence) over PCIe instead"}
    del uh, img

    # ---- the data loader's up-sampling pre-stage (SURVEY 8 a13), reported beside the headline ----
    pre_stage = None
    if rank == 0 and world == 1:
        from skeleton_action_recognition_b200 import pad_frames
        pn, pk = props.multi_processor_count, 250               # one (sequence, coordinate) plane per CTA, 3 waves
        px = synth_batch(pn, 99).to(dev)
        po = torch.empty(pn, 3, T * pk, V, M, device=dev)
        pms = timed(lambda: pad_frames(px, pk, out=po), 5)
        pbytes = po.numel() * 4 + px.numel() * 4
        pre_stage = {"op": "pad_frames (Dataset.pad_frames + cast, utils.py:128-140), num_pad_frames=250, sigma=3",
                     "n": pn, "ms": pms, "value": pn / (pms * 1e-3), "unit": "sequences/s",
                     "hbm_achieved_gbs": pbytes / (pms * 1e-3) / 1e9, "hbm_frac": pbytes / (pms * 1e-3) / 1e9 / peak,
                     "bytes_per_sequence": pbytes // pn}
        if not args.no_cpu_baseline:
            from oracle import pad_frames as opf
            t0 = time.perf_counter()
            opf.dataset_getitem(px[0].cpu().numpy(), pk)
            dt1 = time.perf_counter() - t0
            pre_stage["cpu_baseline"] = {"value": 1.0 / dt1, "unit": "sequences/s", "cores": 1, "kind": "port",
                                         "sample": "one sequence through scipy gaussian_filter1d + interp1d (%.2f s)" % dt1}
        del px, po

    # ---- the rows next to the headline path (SURVEY 8f): fused consumer resize, fused up-sampling ----
    next_rows = None
    train_step = None
    if rank == 0 and world == 1:
        img_n = 4096
        xi = xb[:img_n]
        ms_f = timed(lambda: layer.forward_image(xi, S), 20)
        ms_u = timed(lambda: torch.nn.functional.interpolate(layer(xi).unsqueeze(1), S), 20)
        img_bytes = BYTES_IN + 4 * S * S
        next_rows = {"consumer_stage": {
            "op": "VirtualRadar + unsqueeze + nearest interpolate to 256x256 (models/resnet.py:24-26) in one launch",
            "n": img_n, "ms": ms_f, "value": img_n / (ms_f * 1e-3), "unit": "sequences/s",
            "hbm_achieved_gbs": img_bytes * img_n / (ms_f * 1e-3) / 1e9, "hbm_frac": img_bytes * img_n / (ms_f * 1e-3) / 1e9 / peak,
            "bytes_per_sequence": img_bytes, "two_launch_ms": ms_u, "speedup_vs_two_launches": ms_u / ms_f}}
        from skeleton_action_recognition_b200 import pad_frames as _pf
        ux = synth_batch(un, 55).to(dev)
        ubuf = torch.empty(un, 3, T * uk, V, M, device=dev)
        ms_f = timed(lambda: layer.forward_upsampled(ux, uk, 3, image_size=S), 3)
        ms_u = timed(lambda: layer.forward_image(_pf(ux, uk, 3, out=ubuf), S), 3)
        next_rows["upsampled_pipeline"] = {
            "op": "Dataset.pad_frames(250, sigma 3) + cast + VirtualRadar + resize (utils.py:128-140, models/resnet.py:23-26): "
                  "spline solve + one fused launch, the 45 MB/sequence up-sampled batch never exists",
            "n": un, "frames_per_sequence": T * uk, "ms": ms_f, "value": un / (ms_f * 1e-3), "unit": "sequences/s",
            "two_launch_ms": ms_u, "two_launch_value": un / (ms_u * 1e-3), "speedup_vs_two_launches": ms_u / ms_f,
            "fp32_tflops": (55 * T * uk * 24 * M) * un / (ms_f * 1e-3) / 1e12}
        del ux, ubuf

        # ---- BASELINE configs 1 and 3: the notebook's single long sequences (cells 4 / 2 / 3), synthetic data of the same
        # shape, dtype and bone lists: raw (T, V, 3) array on the device -> utils.pad_frames on the device -> radar ------
        gait_edges = [(0, 1), (1, 2), (1, 3), (3, 5), (5, 7), (1, 4), (4, 6), (6, 8), (0, 9),
                      (9, 11), (11, 13), (13, 15), (0, 10), (10, 12), (12, 14), (14, 16)]
        nb_cases = (("config1_ntu_x550", 300, 25, 550, torch.float32, None, 9e-4),
                    ("config3_cmu_x20", 2751, 42, 20, torch.float64, [(i, i + 1) for i in range(41)], 5e-3),
                    ("config3_gait_x10", 8192, 17, 10, torch.float64, gait_edges, 5e-4))
        notebook = {"op": "virtual_radar_example.ipynb cells 2-4 on the device: pad_frames (utils.py:82-89) + VirtualRadar.forward "
                          "(VirtualRadar.forward_notebook: two launches), one sequence, synthetic smooth motion of the notebook's shapes"}
        for name, t_raw, v_n, kpad, dt, eds, lam in nb_cases:
            gq = torch.Generator().manual_seed(t_raw)
            tt = torch.linspace(0, 6.28, t_raw, dtype=torch.float64)[:, None, None]
            raw = (torch.randn(1, v_n, 3, generator=gq, dtype=torch.float64) * 0.3
                   + 0.1 * torch.sin(tt * (1 + torch.arange(v_n, dtype=torch.float64)[None, :, None] / v_n))).to(dt)
            kw = dict(wavelength=lam, device=dev)
            if eds is not None:
                kw["edges"] = eds
            lay = VirtualRadar(**kw).to(dev)
            rd = raw.to(dev)
            ms_nb = timed(lambda: lay.forward_notebook(rd, kpad), 10)
            entry = {"raw_frames": t_raw, "joints": v_n, "frames_at_radar_rate": t_raw * kpad, "ms": ms_nb,
                     "out_shape": [1, N_FFT, t_raw * kpad // HOP + 1]}
            if name == "config1_ntu_x550" and not args.no_cpu_baseline:
                from oracle import pad_frames as opf2, virtual_radar_oracle as vro2
                t0 = time.perf_counter()
                xo = opf2.notebook_tensor(opf2.pad_frames(raw.numpy(), num_pad_frames=kpad))
                vro2.forward(xo, wavelength=lam)
                dtc = time.perf_counter() - t0
                entry["cpu_baseline"] = {"value": dtc * 1e3, "unit": "ms", "cores": torch.get_num_threads(), "kind": "port",
                                         "sample": "scipy pad_frames + the reference's forward (oracle port), once"}
            notebook[name] = entry
            del lay, rd
        next_rows["notebook_configs"] = notebook

        # ---- BASELINE config 5: the consumer's training step with the fused input stage ----------
        from skeleton_action_recognition_b200.models.resnet import Model
        tb = 64
        labels = torch.randint(0, 60, (tb,), generator=torch.Generator().manual_seed(1)).to(dev)
        train_step = {"op": "main_spectrogram.py:146-158: outputs = model(inputs); CrossEntropyLoss; backward; Adam step -- "
                            "Model = VirtualRadar input stage + ResNet-18 (reference layout: 1 input channel, 64 filters, 60 classes), "
                            "batch 64, image 256x256, float32, random-init weights, synthetic labels; the classifier is stock PyTorch/cuDNN",
                      "batch": tb}
        for name, kpad in (("radar_rate_input", None), ("raw_input_upsampled_x250", 250)):
            model = Model(num_classes=60, num_filters=64, image_size=256, device=dev, num_pad_frames=kpad).to(dev)
            opt = torch.optim.Adam(model.parameters(), lr=1e-3)
            xt = synth_batch(tb, 7).to(dev)

            def one_step():
                opt.zero_grad(set_to_none=True)
                loss = torch.nn.functional.cross_entropy(model(xt), labels)
                loss.backward()
                opt.step()
                return loss
            ms_step = timed(one_step, 10)
            with torch.no_grad():
                ms_in = timed(lambda: model.spectrogram_image(xt), 10)
            train_step[name] = {"ms_per_step": ms_step, "samples_per_s": tb / (ms_step * 1e-3),
                                "input_stage_ms": ms_in, "input_stage_share": ms_in / ms_step,
                                "input_frames_per_sequence": T * (kpad or 1)}
            del model, opt, xt
    del xb

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        times = time_cpu_port(BATCH, 3)
        cpu_baseline = {"value": BATCH / min(times), "unit": "spectrograms/s", "cores": torch.get_num_threads(),
                        "kind": "port", "sample": "the full N=256 batch once per repeat, best of 3 (%.2f s each)" % min(times)}

    if rank == 0:
        traffic, traffic_src = ncu_traffic("dram_bytes_per_launch_n256")
        line = {
            "metric": "spectrograms/sec (NTU 3x300x25x2)", "value": value, "unit": "spectrograms/s",
            "n_gpus": world, "steps": K, "warmup": warm_n, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "batch_per_gpu": BATCH, "sharding": "by sequence, no collective on the path",
                       "l2": "steps rotate over %d input/output buffer pairs (%.0f MB > 126 MB L2)" % (pool, pool * BATCH * BYTES_PER_SPEC / 1e6),
                       "timing": "one window of exactly %d steps between CUDA events, max over ranks, after %d warm-up steps "
                                 "(>= --warmup %d, launched over >= %.0f ms)" % (K, warm_n, args.warmup, MIN_WARM_MS),
                       "launch": {"cooperative": plan, "team_jobs": plan_team,
                                  "schedule": "team jobs for overlapping or large batches, cooperative otherwise (vr_set_schedule)"},
                       "overlap": "value: steps are independent batches, programmatic dependent launches with VR_FLAG_INPUTS_READY "
                                  "(a step's reads may start while the previous step's last CTAs finish; writes wait); "
                                  "stream_ordered: the same loop without the flag, the module's default"},
            "stream_ordered": {"value": world * BATCH / (so_ms * 1e-3), "ms_per_step": so_ms, "steps": K, "warmup": so_warm,
                               "hbm_frac": frac(BATCH, so_ms),
                               "note": "same loop without the flag: every step waits for the previous kernel to finish"},
            "module_forward": module_forward,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": BYTES_PER_SPEC * BATCH,
                         "fp32_tflops": FLOPS_PER_SPEC * BATCH / (ms_per_step * 1e-3) / 1e12,
                         "fp32_frac_of_derived_peak": FLOPS_PER_SPEC * BATCH / (ms_per_step * 1e-3) / 1e12 / fp32_peak},
            "large_batch": {"n_per_gpu": big_n, "value": big_value, "ms_per_launch": big_ms,
                            "hbm_achieved_gbs": big_achieved, "hbm_frac": big_achieved / peak,
                            "note": "one stream-ordered launch over 16384 sequences per GPU (2.95 GB in, 0.32 GB out)"},
            "sweep": {"what": "BASELINE config 4: global batch sharded by sequence over %d rank(s), stream-ordered launches, aggregate sequences/s" % world,
                      "points": sweep},
            "e2e": {"value": e2e_value, "unit": "spectrograms/s", "h2d_bytes_per_step": BATCH * BYTES_IN,
                    "d2h_bytes_per_step": BATCH * BYTES_OUT, "steps": e2e_steps,
                    "api": "VirtualRadar.forward_host (C ABI vr_forward_host_f32), pinned host buffers"},
            "e2e_upsampled": e2e_upsampled,
            "gpu_launches": K,
            "source_hash": source_hash(),
            "clocks": sampler.summary(),
        }
        for key, val in (("shard_verify", shard_verify), ("cpu_baseline", cpu_baseline), ("pre_stage", pre_stage),
                         ("next_rows", next_rows), ("train_step", train_step)):
            if val:
                line[key] = val
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the spectrograms of the last timed step to DIR/spectrograms.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world == 1 and args.gpus > 1 and args.impl == "ours":
        # convenience: relaunch under torchrun, with every argument of this call
        import subprocess
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", "29517", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    # exactly ONE line on stdout: libraries (NCCL's version banner, torch warnings) write to fd 1 too, so
    # everything except the final JSON line is sent to stderr
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = real_stdout
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)
    real_stdout.flush()


if __name__ == "__main__":
    main()
