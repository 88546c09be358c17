"""ctypes binding of include/virtual_radar_b200.h (libvirtual_radar_b200.so, built in-tree by
__graft_entry__.build()).  There is deliberately no fallback: if the shared object is missing the
import of the layer fails loudly."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libvirtual_radar_b200.so")

VR_OK, VR_ERR_ARG, VR_ERR_SHAPE, VR_ERR_UNSUPPORTED, VR_ERR_CUDA = 0, -1, -2, -3, -4
VR_FLAG_RANGE_FMA = 1
VR_FLAG_INPUTS_READY = 2
VR_FLAG_PER_SEQUENCE = 4
VR_FLAG_NOISE = 8               # receiver noise from vr_set_noise (with VR_FLAG_PER_SEQUENCE); never passed to a backward entry
VR_FLAG_VIEWS_SHIFT = 8         # VR_FLAG_VIEWS(R) = R << 8, R in [1, 255]: R radars per sequence (with VR_FLAG_PER_SEQUENCE)
VR_FLAG_VIEWS_MASK = 0xff << VR_FLAG_VIEWS_SHIFT
ABI_VERSION = 1

# every symbol include/virtual_radar_b200.h declares
SYMBOLS = ("vr_abi_version", "vr_last_error", "vr_forward_f32", "vr_forward_debug_f32",
           "vr_forward_host_f32", "vr_release_host_staging", "vr_plan", "vr_partition_edges",
           "vr_set_tuning", "vr_selftest_rounding", "vr_set_timeline_buffer", "vr_pad_frames_f32",
           "vr_forward_image_f32", "vr_plan_image", "vr_forward_upsampled_f32", "vr_upsampled_workspace_bytes", "vr_backward_params_f32", "vr_backward_f32", "vr_synth_adjoint_f32", "vr_job_geometry",
           "vr_set_schedule", "vr_plan_team", "vr_pad_frames_joints",
           "vr_pad_frames_backward_f32", "vr_forward_upsampled_debug_f32", "vr_backward_upsampled_params_f32",
           "vr_stft_general_workspace_floats", "vr_stft_general_f32", "vr_stft_general_backward_f32",
           "vr_synth_f32", "vr_synth_upsampled_f32", "vr_synth_adjoint_upsampled_f32",
           "vr_stft_general_frames_workspace_floats", "vr_stft_general_frames_f32", "vr_stft_general_frames_backward_f32",
           "vr_plan_adjoint_stft", "vr_plan_pad_frames", "vr_plan_stft_general", "vr_per_sequence_grad_doubles",
           "vr_set_noise", "vr_plan_launch", "vr_plan_backward")

_lib = None


class VirtualRadarLibraryError(ImportError):
    pass


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise VirtualRadarLibraryError(
            "%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). There is no CPU or PyTorch fallback for VirtualRadar." % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    c_i32p = ctypes.POINTER(ctypes.c_int32)
    vp, i64, i32, u32, f32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_uint32, ctypes.c_float
    L.vr_abi_version.restype = ctypes.c_int
    L.vr_last_error.restype = ctypes.c_char_p
    common = [vp, i64, i64, i32, i32, c_i32p, c_i32p, i32]
    L.vr_forward_f32.argtypes = common + [vp, vp, i32, i32, u32, vp, vp]
    L.vr_forward_debug_f32.argtypes = common + [vp, vp, i32, i32, u32, vp, vp, vp]
    L.vr_forward_image_f32.argtypes = common + [vp, vp, i32, i32, u32, i32, vp, vp]
    L.vr_forward_upsampled_f32.argtypes = common + [vp, vp, i32, i32, u32, i32, f32, i32, vp, i64, vp, vp]
    L.vr_forward_upsampled_f32.restype = ctypes.c_int
    L.vr_forward_upsampled_debug_f32.argtypes = common + [vp, vp, i32, i32, u32, i32, f32, vp, i64, vp, vp, vp]
    L.vr_forward_upsampled_debug_f32.restype = ctypes.c_int
    L.vr_backward_upsampled_params_f32.argtypes = [vp, vp, vp, i64, i64, i32, i32, c_i32p, c_i32p, i32, vp, vp, i32, i32, u32,
                                                   i32, vp, vp, vp]
    L.vr_backward_upsampled_params_f32.restype = ctypes.c_int
    L.vr_synth_f32.argtypes = common + [vp, vp, u32, vp, vp]
    L.vr_synth_f32.restype = ctypes.c_int
    L.vr_synth_upsampled_f32.argtypes = common + [vp, vp, u32, i32, f32, vp, i64, vp, vp]
    L.vr_synth_upsampled_f32.restype = ctypes.c_int
    L.vr_synth_adjoint_upsampled_f32.argtypes = [vp, vp, i64, i64, i32, i32, c_i32p, c_i32p, i32, vp, vp, u32, i32, vp, vp]
    L.vr_synth_adjoint_upsampled_f32.restype = ctypes.c_int
    L.vr_upsampled_workspace_bytes.argtypes = [i64, i64, i32, i32]
    L.vr_upsampled_workspace_bytes.restype = i64
    L.vr_backward_params_f32.argtypes = [vp, vp, vp, i64, i64, i32, i32, c_i32p, c_i32p, i32, vp, vp, i32, i32, u32, vp, vp, vp]
    L.vr_backward_params_f32.restype = ctypes.c_int
    L.vr_backward_f32.argtypes = [vp, vp, vp, i64, i64, i32, i32, c_i32p, c_i32p, i32, vp, vp, i32, i32, u32, vp, vp, vp, vp]
    L.vr_backward_f32.restype = ctypes.c_int
    L.vr_synth_adjoint_f32.argtypes = [vp, vp, i64, i64, i32, i32, c_i32p, c_i32p, i32, vp, vp, u32, vp, vp, vp]
    L.vr_synth_adjoint_f32.restype = ctypes.c_int
    L.vr_job_geometry.argtypes = [i64, i64, i32, i32, c_i32p, c_i32p, i32, i32, i32, i32, i64, ctypes.POINTER(i64)]
    L.vr_job_geometry.restype = ctypes.c_int
    L.vr_plan_image.argtypes = [i64, i64, i32, i32, c_i32p, c_i32p, i32, i32, i32, i32, i32, ctypes.POINTER(i64)]
    L.vr_forward_host_f32.argtypes = common + [f32, ctypes.POINTER(f32), i32, i32, u32, vp, i64]
    L.vr_plan.argtypes = [i64, i64, i32, i32, c_i32p, c_i32p, i32, i32, i32, i32, ctypes.POINTER(i64)]
    L.vr_partition_edges.argtypes = [c_i32p, c_i32p, i32, i32, c_i32p]
    L.vr_set_tuning.argtypes = [ctypes.c_int] * 3
    L.vr_plan_team.argtypes = [i64, i64, i32, i32, c_i32p, c_i32p, i32, i32, i32, i32, ctypes.POINTER(i64)]
    L.vr_plan_team.restype = ctypes.c_int
    L.vr_set_schedule.argtypes = [ctypes.c_int]
    L.vr_set_schedule.restype = ctypes.c_int
    L.vr_pad_frames_f32.argtypes = [vp, i64, i64, i32, i32, i32, f32, vp, vp]
    L.vr_pad_frames_f32.restype = ctypes.c_int
    L.vr_pad_frames_backward_f32.argtypes = [vp, i64, i64, i32, i32, i32, f32, vp, vp]
    L.vr_pad_frames_backward_f32.restype = ctypes.c_int
    L.vr_pad_frames_joints.argtypes = [vp, i32, i64, i64, i32, i32, i32, f32, i32, vp, vp]
    L.vr_pad_frames_joints.restype = ctypes.c_int
    L.vr_stft_general_workspace_floats.argtypes = [i64, i64, i32, i32, ctypes.POINTER(i64)]
    L.vr_stft_general_workspace_floats.restype = i64
    L.vr_stft_general_f32.argtypes = [vp, i64, i64, i32, i32, vp, vp, vp, vp, vp, vp, vp]
    L.vr_stft_general_f32.restype = ctypes.c_int
    L.vr_stft_general_backward_f32.argtypes = [vp, vp, vp, vp, i64, i64, i32, i32, vp, vp, vp, vp, vp, vp, vp]
    L.vr_stft_general_backward_f32.restype = ctypes.c_int
    L.vr_stft_general_frames_workspace_floats.argtypes = [i64, i64, i32, ctypes.POINTER(i64)]
    L.vr_stft_general_frames_workspace_floats.restype = i64
    L.vr_stft_general_frames_f32.argtypes = [vp, i64, i64, i32, i32, vp, i64, vp, vp, vp, vp, vp, vp, vp]
    L.vr_stft_general_frames_f32.restype = ctypes.c_int
    L.vr_stft_general_frames_backward_f32.argtypes = [vp, vp, vp, vp, i64, i64, i32, i32, vp, i64, vp, vp, vp, vp, vp, vp, vp]
    L.vr_stft_general_frames_backward_f32.restype = ctypes.c_int
    L.vr_plan_adjoint_stft.argtypes = [i64, i64, i32, i32, ctypes.POINTER(i64), ctypes.POINTER(i64), i64]
    L.vr_plan_adjoint_stft.restype = ctypes.c_int
    L.vr_plan_pad_frames.argtypes = [i32, i64, i64, i32, i32, i32, f32, i32, ctypes.POINTER(i64)]
    L.vr_plan_pad_frames.restype = ctypes.c_int
    L.vr_plan_stft_general.argtypes = [i64, i64, i32, i32, i64, i32, ctypes.POINTER(i64)]
    L.vr_plan_stft_general.restype = ctypes.c_int
    L.vr_per_sequence_grad_doubles.argtypes = [i64, i64]
    L.vr_per_sequence_grad_doubles.restype = i64
    L.vr_plan_launch.argtypes = [i32, i64, i64, i32, i32, c_i32p, c_i32p, i32, i32, i32, i32, i32, u32, i32, i32, i32,
                                 ctypes.POINTER(i64)]
    L.vr_plan_launch.restype = ctypes.c_int
    L.vr_plan_backward.argtypes = [i32, i64, i64, i32, i32, c_i32p, c_i32p, i32, i32, i32, u32, i32, i32, i32,
                                   ctypes.POINTER(i64)]
    L.vr_plan_backward.restype = ctypes.c_int
    L.vr_set_noise.argtypes = [vp, vp]
    L.vr_set_noise.restype = ctypes.c_int
    L.vr_set_timeline_buffer.argtypes = [vp]
    L.vr_set_timeline_buffer.restype = ctypes.c_int
    L.vr_selftest_rounding.argtypes = [ctypes.c_uint64, f32, ctypes.POINTER(ctypes.c_uint64)]
    L.vr_selftest_rounding.restype = ctypes.c_int
    for name in ("vr_forward_f32", "vr_forward_debug_f32", "vr_forward_host_f32", "vr_plan", "vr_forward_image_f32", "vr_plan_image",
                 "vr_partition_edges", "vr_set_tuning", "vr_release_host_staging"):
        getattr(L, name).restype = ctypes.c_int
    if L.vr_abi_version() != ABI_VERSION:
        raise VirtualRadarLibraryError("ABI mismatch: library %d, binding %d" % (L.vr_abi_version(), ABI_VERSION))
    _lib = L
    return L


def last_error():
    return lib().vr_last_error().decode("utf-8", "replace")


def check(rc):
    """Map a VR_ERR_* code to the exception class the reference would raise in that situation."""
    if rc == VR_OK:
        return
    msg = last_error()
    if rc in (VR_ERR_ARG, VR_ERR_SHAPE):
        raise ValueError(msg)
    if rc == VR_ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise RuntimeError(msg)


def i32_array(values):
    arr = (ctypes.c_int32 * len(values))(*[int(v) for v in values])
    return arr


PLAN_FIELDS = ("grid", "block", "smem_bytes", "ring_stages", "frames_per_job", "jobs_per_seq",
               "frames_per_tile", "tma_loads", "tma_bulk_store", "chunks_per_job", "max_bones_per_group",
               "max_sources_per_group", "z_capacity", "ctas_per_sm", "chunk_steps", "lane_groups")


def plan(N, T, V, M, src, dst, n_fft=256, hop=16, sm_count=148):
    out = (ctypes.c_int64 * 16)()
    check(lib().vr_plan(N, T, V, M, i32_array(src), i32_array(dst), len(src), n_fft, hop, sm_count, out))
    return dict(zip(PLAN_FIELDS, [int(v) for v in out]))


IMAGE_PLAN_FIELDS = PLAN_FIELDS[:4] + ("columns_per_job",) + PLAN_FIELDS[5:10] + ("sparse_frames", "columns") + PLAN_FIELDS[12:]


def plan_image(N, T, V, M, src, dst, image_size, n_fft=256, hop=16, sm_count=148):
    out = (ctypes.c_int64 * 16)()
    check(lib().vr_plan_image(N, T, V, M, i32_array(src), i32_array(dst), len(src), n_fft, hop, image_size, sm_count, out))
    return dict(zip(IMAGE_PLAN_FIELDS, [int(v) for v in out]))


TEAM_PLAN_FIELDS = ("grid", "block", "smem_bytes", "ring_stages_per_team", "teams_per_cta", "stage_bytes", "z_stride", "automatic")


def plan_team(N, T, V, M, src, dst, n_fft=256, hop=16, sm_count=148):
    out = (ctypes.c_int64 * 8)()
    check(lib().vr_plan_team(N, T, V, M, i32_array(src), i32_array(dst), len(src), n_fft, hop, sm_count, out))
    return dict(zip(TEAM_PLAN_FIELDS, [int(v) for v in out]))


LAUNCH_PLAN_FIELDS = ("team", "grid", "block", "smem_bytes", "ring_stages", "columns_per_job", "jobs_per_seq", "jobs",
                      "columns_per_tile", "tile_stride", "tma_loads", "tma_bulk_store", "chunks_per_job", "z_capacity",
                      "parked_sums", "sparse_frames", "columns", "ctas_per_sm", "ticket", "bodies_per_pass", "compiled_vm",
                      "max_bones_per_group", "max_sources_per_group", "iq_fill")
LAUNCH_MODES = {"spectrogram": 0, "debug": 1, "synth": 2}


def plan_launch(mode, N, T, V, M, src, dst, hop=16, image_size=0, num_pad_frames=0, flags=0, x_aligned=True, schedule=-1,
                sm_count=148, n_fft=256):
    """Configuration of one fused forward launch (vr_plan_launch): mode "spectrogram" (vr_forward_f32, _image_f32 with
    image_size, _upsampled_f32 with num_pad_frames and T raw), "debug" (the entries that write iq as well) or "synth"
    (synthesis only); schedule as set_schedule."""
    out = (ctypes.c_int64 * len(LAUNCH_PLAN_FIELDS))()
    check(lib().vr_plan_launch(LAUNCH_MODES[mode], N, T, V, M, i32_array(src), i32_array(dst), len(src), n_fft, hop,
                               image_size, num_pad_frames, flags, 1 if x_aligned else 0, schedule, sm_count, out))
    return dict(zip(LAUNCH_PLAN_FIELDS, [int(v) for v in out]))


ADJOINT_PLAN_FIELDS = ("segment_length", "segments", "grid", "smem_bytes")


def plan_adjoint_stft(N, T, hop=16, sm_count=148):
    """The owner-form plan of the adjoint STFT -> (plan dict, [(first sample, end sample, first frame, last frame)] per
    segment of a sequence)."""
    out = (ctypes.c_int64 * 4)()
    check(lib().vr_plan_adjoint_stft(N, T, hop, sm_count, out, None, 0))
    plan = dict(zip(ADJOINT_PLAN_FIELDS, [int(v) for v in out]))
    rows = (ctypes.c_int64 * (4 * plan["segments"]))()
    check(lib().vr_plan_adjoint_stft(N, T, hop, sm_count, out, rows, plan["segments"]))
    return plan, [tuple(int(v) for v in rows[4 * k:4 * k + 4]) for k in range(plan["segments"])]


BACKWARD_PLAN_FIELDS = ("stft", "segment_length", "segments", "stft_grid", "stft_smem_bytes", "synth_kernel", "ups",
                        "views_mode", "views", "grid", "units", "ps_segments", "fold_grid", "scratch_tail", "grad_x_fill",
                        "grid_cap")
BACKWARD_ENTRIES = {"backward": 0, "backward_params": 1, "synth_adjoint": 2, "backward_upsampled_params": 3,
                    "synth_adjoint_upsampled": 4}
SYNTH_KERNELS = ("scalar", "scalar_ups", "ps")
VIEWS_MODES = ("none", "outputs", "rows")


def plan_backward(entry, N, T, V, M, src, dst, hop=16, flags=0, grad_x=False, num_pad_frames=0, sm_count=148, n_fft=256):
    """Configuration of one backward call (vr_plan_backward): entry "backward" (vr_backward_f32), "backward_params",
    "synth_adjoint", "backward_upsampled_params" or "synth_adjoint_upsampled" (T raw, with num_pad_frames); grad_x: a
    dL/dx buffer is passed.  synth_kernel and views_mode come back as names."""
    out = (ctypes.c_int64 * len(BACKWARD_PLAN_FIELDS))()
    check(lib().vr_plan_backward(BACKWARD_ENTRIES[entry], N, T, V, M, i32_array(src), i32_array(dst), len(src), n_fft, hop,
                                 flags, 1 if grad_x else 0, num_pad_frames, sm_count, out))
    plan = dict(zip(BACKWARD_PLAN_FIELDS, [int(v) for v in out]))
    plan["synth_kernel"] = SYNTH_KERNELS[plan["synth_kernel"]]
    plan["views_mode"] = VIEWS_MODES[plan["views_mode"]]
    return plan


PAD_PLAN_FIELDS = ("nc", "ncb", "units", "grid", "smem_bytes", "nrs", "rows_per_slice", "radius")
PAD_KINDS = {"forward": 0, "backward": 1, "notebook": 2}


def plan_pad_frames(kind, N, T, V, M_or_C, num_pad_frames, sigma, sm_count=148):
    """Launch configuration of vr_pad_frames_f32 ("forward"), vr_pad_frames_backward_f32 ("backward") or
    vr_pad_frames_joints ("notebook", M_or_C = C)."""
    out = (ctypes.c_int64 * 8)()
    check(lib().vr_plan_pad_frames(PAD_KINDS[kind], N, T, V, M_or_C, num_pad_frames, ctypes.c_float(float(sigma)),
                                   sm_count, out))
    return dict(zip(PAD_PLAN_FIELDS, [int(v) for v in out]))


STFT_PLAN_FIELDS = ("nb", "F", "M", "ldm", "Lp", "row_tiles", "col_tiles", "kblocks", "dbt_tiles", "splits", "kb_per_split",
                    "kb_last", "hop_view")


def plan_stft_general(N, T, n_fft, hop, F_kept=0, sm_count=148):
    """Launch configuration of the general-kernel STFT's GEMMs (vr_stft_general_f32 and its backward; F_kept > 0: the
    kept-frames entries)."""
    out = (ctypes.c_int64 * len(STFT_PLAN_FIELDS))()
    check(lib().vr_plan_stft_general(N, T, n_fft, hop, F_kept, sm_count, out))
    return dict(zip(STFT_PLAN_FIELDS, [int(v) for v in out]))


def per_sequence_grad_doubles(N, T):
    """Length in float64 values of the gradient buffer of a backward call with VR_FLAG_PER_SEQUENCE: N x 4 per-sequence
    gradients, then the scratch of the per-sequence reduction.  T: the steps the adjoint runs over (up-sampled length for
    the _upsampled entries)."""
    return int(lib().vr_per_sequence_grad_doubles(int(N), int(T)))


def views_flag(R):
    """VR_FLAG_VIEWS(R): R radar views per sequence, x holding N / R sequences (add VR_FLAG_PER_SEQUENCE)."""
    R = int(R)
    if not 1 <= R <= 255:
        raise ValueError("the number of views per sequence must be in [1, 255], got %d" % R)
    return R << VR_FLAG_VIEWS_SHIFT


def views_of(flags):
    """R of the VR_FLAG_VIEWS field of `flags` (1 when the field is 0): outputs per x sequence."""
    return ((int(flags) & VR_FLAG_VIEWS_MASK) >> VR_FLAG_VIEWS_SHIFT) or 1


def set_noise(noise_std, seed):
    """vr_set_noise for the next VR_FLAG_NOISE launch of this thread: noise_std (N,) float32 and seed, a 0-d int64 tensor
    holding the 64 seed bits, both on the launch's device (contiguous)."""
    check(lib().vr_set_noise(noise_std.data_ptr(), seed.data_ptr()))


def set_schedule(mode):
    """-1 automatic (default), 0 cooperative kernel only, 1 team-job kernel whenever the shape qualifies."""
    check(lib().vr_set_schedule(int(mode)))


GEOM_FIELDS = ("sequence", "first_column", "columns", "first_frame", "frames", "lo", "hi", "chunks")


def job_geometry(N, T, V, M, src, dst, job, image_size=0, n_fft=256, hop=16):
    out = (ctypes.c_int64 * 8)()
    check(lib().vr_job_geometry(N, T, V, M, i32_array(src), i32_array(dst), len(src), n_fft, hop, image_size, job, out))
    return dict(zip(GEOM_FIELDS, [int(v) for v in out]))


def selftest_rounding(n, wavelength):
    out = (ctypes.c_uint64 * 3)()
    check(lib().vr_selftest_rounding(n, wavelength, out))
    return [int(v) for v in out]


def partition_edges(src, dst, V):
    out = (ctypes.c_int32 * len(src))()
    check(lib().vr_partition_edges(i32_array(src), i32_array(dst), len(src), V, out))
    return [int(v) for v in out]
